"""Host-side logic of bench.py that does not need a GPU: the roofline post-processing of the library's profile report,
the CPU budget probe and the argument defaults the driver relies on."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)

PEAKS = dict(hbm=6574.1, tf=1404.6, src="test")


def fake_prof():
    return {
        "lk_track": {"ms": 40.0, "calls": 100, "work": 100 * 38.0e6},      # 0.4 ms per launch, 38 MB each -> 95 GB/s
        "pyrdown": {"ms": 10.0, "calls": 100, "work": 100 * 45.9e6},
        "imu_cov_propagate": {"ms": 20.0, "calls": 100, "work": 100 * 2.0e6},
        "ekf_gain": {"ms": 6.0, "calls": 100, "work": 0},
        "ekf_cov": {"ms": 2.0, "calls": 100, "work": 0},
        "ekf_update": {"ms": 0.0, "calls": 0, "work": 100 * 64 * 4.4e6},   # Joseph flops attributed to the pair
        "cov_edit": {"ms": 1.0, "calls": 200, "work": 0},
        "host:gating": {"ms": 12.0, "calls": 100},
        "_h2d_bytes": 1.0e9,
        "_d2h_bytes": 1.0e8,
    }


def test_roofline_picks_dominant_kernel_and_computes_achieved():
    r, host = bench.build_roofline(fake_prof(), K=25, peaks=PEAKS, seqs_per_launch=64, pass_ms=60.0)
    assert r["kernel"] == "lk_track" and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert abs(r["achieved"] - 38.0e6 / 0.4e-3 / 1e9) < 1e-9 and abs(r["frac"] - r["achieved"] / PEAKS["hbm"]) < 1e-12
    assert r["launches"] == 100 and abs(r["avg_launch_us"] - 400.0) < 1e-9
    assert abs(sum(v["share"] for v in r["kernels"].values()) - 1.0) < 1e-3
    assert "ekf_gain" not in r["kernels"] and abs(r["kernels"]["ekf_update"]["ms"] - 8.0) < 1e-9  # gain + cov merged
    assert abs(r["device_busy_frac"] - 79.0 / 60.0) < 1e-9 and abs(r["profiled_pass_ms_per_step"] - 2.4) < 1e-12
    assert host == {"gating": 0.48}
    # EKF-update time per frame (BASELINE.json's second figure): (6 + 2) ms over 100 launches of 64 filters
    assert r["ekf_update"]["us_per_launch"] == 80.0 and abs(r["ekf_update"]["us_per_frame"] - 1.25) < 1e-9 and r["ekf_update"]["filters_per_launch"] == 64
    pk = r["per_kernel"]
    assert set(pk) == {"lk_track", "pyrdown", "imu_cov_propagate", "ekf_update"}
    assert pk["ekf_update"]["bound"] == "tensor" and abs(pk["ekf_update"]["achieved"] - 100 * 64 * 4.4e6 / 8e-3 / 1e12) < 1e-3
    assert r["traffic"] is None or r["traffic"] > 0  # profiles/r01_traffic.json scaled to 64 sequences per launch
    json.dumps(r)  # serialisable


def test_roofline_tensor_bound_when_update_dominates_and_empty_report():
    p = fake_prof()
    p["ekf_gain"]["ms"] = 500.0
    r, _ = bench.build_roofline(p, 25, PEAKS, 64, 600.0)
    assert r["kernel"] == "ekf_update" and r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and r["peak"] == PEAKS["tf"]
    r, host = bench.build_roofline({"_h2d_bytes": 0, "_d2h_bytes": 0}, 25, PEAKS, 64, 1.0)
    assert r["kernel"] is None and host == {}


def test_cpu_budget_is_positive_and_bounded_by_affinity():
    n = bench.cpu_budget()
    assert 1 <= n <= len(os.sched_getaffinity(0))


def test_defaults_match_the_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert r.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--seqs", "--batches", "--cov-update"):
        assert flag in r.stdout
    assert bench.measured_peaks()["hbm"] > 1000


def test_cpu_baseline_entry_kinds():
    r = dict(fps=4000.0, mean_frame_ms=4.0, stage_share=dict(lk=0.7, fast=0.2, gate=0.02, update=0.08), eigen=True, fps_reference=None)
    e = bench.cpu_baseline_entry(r, 16, 80, 12.0)
    assert e["kind"] == "port" and e["value"] == 4000.0 and e["cores"] == 16
    r.update(fps_reference=2900.0, tracker_ms=3.2, ref_estimator_ms=2.9, ref_tracks=150.0)
    e = bench.cpu_baseline_entry(r, 16, 80, 12.0)
    assert e["kind"] == "reference" and e["value"] == 2900.0 and e["numerics_only_value"] == 4000.0 and "reference's own" in e["sample"]
    json.dumps(e)


def test_cpu_baseline_runs_the_reference_library_when_it_is_built():
    """oracle/cpu_baseline.py end to end on 2 processes x 6 frames: cv2 tracker timing + (where oracle/_ref is built) the reference's own
    estimator on a point-cloud stream -> fps_reference below the numerics-only upper bound."""
    r = subprocess.run([sys.executable, "-m", "oracle.cpu_baseline", os.path.join(ROOT, "xivo_b200", "cfg", "vio_640x480.json"), "2", "6", "13", "4", "14"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["fps"] > 0 and d["frames"] >= 4 and d["cv2"]
    from oracle import ref_runner

    if ref_runner.available(4, 14):
        assert d["fps_reference"] and 0 < d["fps_reference"] < d["fps"] and 0.5 < d["ref_estimator_ms"] < 50 and d["ref_tracks"] == 150
    else:
        assert d["fps_reference"] is None


def test_pick_ingest_keeps_the_default_unless_clearly_faster():
    assert bench.pick_ingest({"copy_engine": [8.4, 8.3], "zero_copy": [8.2, 8.25]}) == "copy_engine"   # 1 % is noise
    assert bench.pick_ingest({"copy_engine": [8.4, 8.3], "zero_copy": [6.1, 6.4]}) == "zero_copy"
    assert bench.pick_ingest({"copy_engine": [6.0, 6.2], "zero_copy": [9.0, 8.8]}) == "copy_engine"
    assert set(bench.INGEST_MODES.values()) == {0, 1}


def test_ingest_calibration_protocol():
    """calibrate_ingest with fakes: every mode is tried in every round, the frames it consumes are exactly the extra frames run_ours renders,
    the winner is left switched on, and a forced mode calibrates nothing."""
    log, frames = [], []
    cost = {0: 0.004, 1: 0.001}  # the copy engine is 4x faster in this fake
    state = {"mode": None}

    def set_mode(m):
        state["mode"] = m
        log.append(m)

    def run_step(k):
        frames.append(k)
        bench.time.sleep(cost[state["mode"]])

    best, table, f_next = bench.calibrate_ingest("auto", set_mode, run_step, lambda: None, 100)
    assert best == "copy_engine" and log[-1] == bench.INGEST_MODES["copy_engine"] and log[:-1] == [0, 1] * bench.CAL_ROUNDS
    assert frames == list(range(100, f_next)) and f_next - 100 == bench.calibration_frames("auto")
    assert set(table) == set(bench.INGEST_MODES) and all(len(v) == bench.CAL_ROUNDS for v in table.values())
    log.clear()
    assert bench.calibrate_ingest("zero_copy", set_mode, run_step, lambda: None, 7) == ("zero_copy", None, 7) and log == [0]
    assert bench.calibration_frames("zero_copy") == 0


def test_config_selection_sets_the_workload_constants():
    """--config 1/2/3 = BASELINE.json configs[1..3]: frame size from the config's camera block, state dimensions as the parity tests use them."""
    import bench

    try:
        for n, (rows, cols, g, f, nstate) in {1: (480, 640, 4, 14, 89), 2: (512, 512, 15, 30, 203), 3: (1024, 1280, 15, 62, 299)}.items():
            c = bench.select_config(n)
            assert (bench.ROWS, bench.COLS, bench.G, bench.F) == (rows, cols, g, f)
            assert 23 + 6 * bench.G + 3 * bench.F == nstate and f"configs[{n}]" in bench.WORKLOAD and c["seqs"] >= 128
            assert bench.load_cfg()["camera_cfg"]["rows"] == rows
    finally:
        bench.select_config(1)


def test_stream_tables_never_hand_one_frame_to_two_sequences_at_the_default_size():
    """bench.py's claim `no two sequences of a GPU read the same frame in the same step` for the default workload (1024 sequences over
    32 base streams, start delays of 3 frames inside a 100-frame period)."""
    import numpy as np

    import bench

    c = bench.CONFIGS[1]
    n, s0 = c["seqs"], c["streams"]
    assert (n // s0) * bench.STAGGER <= bench.PERIOD_FRAMES
    fidx, iidx, base = bench.stream_tables(n, s0, 260)
    key = base[None, :].astype(np.int64) * 100000 + fidx
    for f in range(bench.REST_FRAMES + (n // s0) * bench.STAGGER + 2, 260):  # once every sequence has left its rest phase
        assert len(np.unique(key[f])) == n, f


def test_dump_outputs_writes_every_sequence_in_order(tmp_path):
    """--dump-outputs with stand-in batches (the read-back methods of xivo_b200.pyxivo.Batch): one row per sequence in sequence order
    across batches, finite float arrays only, tracked features padded, the covariance sample seeded, and below 64 MB at every config's default size."""
    import numpy as np

    class FakeBatch:
        def __init__(self, first, N):
            self.first, self.N = first, N

        def gsb(self, s):
            return np.full((3, 4), float(self.first + s))

        def motion(self, s):
            k = float(self.first + s)
            return np.full(3, k), np.full(3, k + 0.1), np.full(3, k + 0.2), np.full((3, 3), k + 0.3)

        def counters(self, s):
            return dict(a=self.first + s, b=7)

        def tracked_features(self, s):
            n = (self.first + s) % 4
            return np.arange(n, dtype=np.int32) + 100, np.full((n, 2), 0.5), np.ones(n, np.int32)

        def P(self, s):
            return np.full((self.N, self.N), float(self.first + s))

    sizes = [30, 20, 20]
    bts = [FakeBatch(0, 5), FakeBatch(30, 5), FakeBatch(50, 5)]
    shapes = bench.dump_outputs(str(tmp_path / "a"), bts, sizes)
    bench.dump_outputs(str(tmp_path / "b"), bts, sizes)
    d = {name: np.load(str(tmp_path / "a" / (name + ".npy"))) for name in shapes}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in d.values())
    assert np.array_equal(d["gsb"][:, 0, 0], np.arange(70)) and np.array_equal(d["Rsg"][:, 2, 2], np.arange(70) + 0.3)
    assert np.array_equal(d["counters"], np.stack([np.arange(70), np.full(70, 7)], 1))
    assert d["tracked_ids"].shape == (70, 3) and d["tracked_ids"][5].tolist() == [100, -1, -1] and (d["tracked_xy"][5, 1:] == -1).all()
    pick = d["P_sample_seqs"].astype(int)
    assert len(pick) == bench.DUMP_P_SEQS and np.array_equal(d["P_sample"][:, 0, 0], pick)
    for name in shapes:  # the same arguments give the same files
        assert np.array_equal(d[name], np.load(str(tmp_path / "b" / (name + ".npy"))))
    try:  # every config at its default size: sequences x (pose, motion, counters, tracked features) + the covariance sample
        for n, c in bench.CONFIGS.items():
            bench.select_config(n)
            tracked = bench.load_cfg()["tracker_cfg"]["num_features_max"]
            N = 23 + 6 * c["G"] + 3 * c["F"]
            assert c["seqs"] * (12 + 18 + 12 + 3 * tracked) * 8 + bench.DUMP_P_SEQS * N * N * 8 < 64 << 20, n
    finally:
        bench.select_config(1)


def test_cpulist_parser_and_numa_placement_is_optional():
    import bench

    assert bench.parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    assert bench.parse_cpulist("") == []
    assert bench.pin_to_gpu_numa_node(0, 1) is None  # no GPU here: placement is skipped, never an error
