#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native XIVO inner loop.

Metric (BASELINE.json): VIO frames/s on synthetic 640x480 + 200 Hz IMU streams, whole job.
Workload (BASELINE.json configs[1]): full VIO, 640x480 pinhole, 150 tracked features, EKF state
dim 89 (G=4, F=14), `--seqs` independent sequences per GPU advancing in lock-step (the filter is
sequential per stream; batching sequences is the only parallel axis — SURVEY.md §8e).  One "step" =
one frame (+ its 8 IMU samples) for every sequence on every GPU.

  python bench.py --gpus N --steps K --warmup W              # this repo (CUDA)
  python bench.py --impl reference --gpus N --steps K --warmup W   # reference CPU arithmetic, all host cores
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + every sequence's state after the last step, DIR/<name>.npy

Prints ONE JSON line (rank 0).  `value` = frames/s with the frames already resident in HBM;
`e2e` = the same through the estimator-level C ABI with pinned HOST frames (H2D inside the timed
region, pose read back every step).  `roofline` describes the kernel with the largest share of
device time (CUDA-event durations recorded by the library on its launch streams) in a third pass over
the next frames of the same streams, in which the batches are stepped one after another so that an
event pair measures the kernel and not the queueing behind other batches' kernels.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS, COLS, G, F = 480, 640, 4, 14
CFG_FILE = "vio_640x480.json"
WORKLOAD = "BASELINE configs[1]: full VIO 640x480 pinhole + 200 Hz IMU, 150 tracked features, state dim 89 (G=4,F=14)"
METRIC = "VIO frames/sec (640x480 synthetic + 200 Hz IMU)"
# --config: the other full-pipeline workloads BASELINE.json names (parity cases of tests/test_gpu_estimator.py); the driver's runs use 1
CONFIGS = {
    1: dict(cfg="vio_640x480.json", G=4, F=14, seqs=1024, streams=32, workload=WORKLOAD, metric=METRIC),  # 1024 x 32: profiles/r02w_sweep.txt
    2: dict(cfg="tumvi_512_equidistant.json", G=15, F=30, seqs=256, streams=8,
            workload="BASELINE configs[2]: TUM-VI equidistant 512x512 + 200 Hz IMU, 200 tracked features, state dim 203 (G=15,F=30)",
            metric="VIO frames/sec (512x512 equidistant synthetic + 200 Hz IMU)"),
    3: dict(cfg="stress_1280x1024.json", G=15, F=62, seqs=128, streams=4,
            workload="BASELINE configs[3]: stress 1280x1024 + 200 Hz IMU, 800 tracked features, state dim 299 (G=15,F=62)",
            metric="VIO frames/sec (1280x1024 synthetic + 200 Hz IMU)"),
}


def select_config(n):
    """Sets the module-level workload constants from CONFIGS[n] (frame size from the config's camera block)."""
    global ROWS, COLS, G, F, CFG_FILE, WORKLOAD, METRIC
    c = CONFIGS[n]
    CFG_FILE, G, F, WORKLOAD, METRIC = c["cfg"], c["G"], c["F"], c["workload"], c["metric"]
    cam = load_cfg()["camera_cfg"]
    ROWS, COLS = int(cam["rows"]), int(cam["cols"])
    return c
IMU_PER_FRAME = 8
FRAME_NS = 40_000_000
PREROLL_FRAMES = 12  # reference arm: gravity init (stationary) + first detections, never timed
CAL_ROUNDS, CAL_STEPS = 2, 4  # frame-ingest calibration: per round and mode one settling step + CAL_STEPS timed steps (untimed region)
INGEST_MODES = {"zero_copy": 0, "copy_engine": 1}


def load_cfg():
    from xivo_b200 import sim

    return sim.load_cfg(os.path.join(ROOT, "xivo_b200", "cfg", CFG_FILE))


ALL_CPUS = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None


def cpu_reference(cores, frames, skip, channels=1):
    """Runs oracle/cpu_baseline.py in a fresh interpreter (no CUDA context there: it forks one worker
    per core) and returns its JSON."""
    cfg_path = os.path.join(ROOT, "xivo_b200", "cfg", CFG_FILE)
    if hasattr(os, "sched_setaffinity"):
        os.sched_setaffinity(0, ALL_CPUS)  # the library pins its driver threads; the CPU arm gets every allowed CPU
    r = subprocess.run([sys.executable, "-m", "oracle.cpu_baseline", cfg_path, str(cores), str(frames), str(skip), str(G), str(F), str(channels)], cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        raise RuntimeError("cpu baseline failed: " + r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d.get("hbm_gbs", 6650.0), tf=d.get("bf16_tflops_sustained", 1400.0), src="MEASURED_PEAKS.json (sustained)")
    return dict(hbm=6650.0, tf=1590.0, src="fallback B200_PROFILING.md")


class ClockSampler:
    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.idx = gpu_index

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i].strip().lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm))


def pick_ingest(ms, default="copy_engine"):
    """ms: {mode: [ms per step of each calibration round]} -> the mode with the best round; the library's default
    (copy_engine) keeps the job unless the alternative is at least 3 % faster (below that it is noise)."""
    best = {k: min(v) for k, v in ms.items() if v}
    if default not in best:
        return min(best, key=best.get)
    alt = min(best, key=best.get)
    return alt if best[alt] < 0.97 * best[default] else default


def calibration_frames(choice):
    """Frames the ingest calibration consumes (run_ours renders that many more)."""
    return CAL_ROUNDS * len(INGEST_MODES) * (1 + CAL_STEPS) if choice == "auto" else 0


def calibrate_ingest(choice, set_mode, run_step, sync, f):
    """Pinned host frames reach the device either by a gather kernel reading host memory over PCIe or by the copy engine
    (xivo_set_frame_ingest); same results, the faster one depends on the host's PCIe path.  Picks per rank, outside every timed
    region, from end-to-end steps of this very workload: per round and mode one settling step + CAL_STEPS timed steps.
    set_mode(int), run_step(frame index), sync() are the caller's; returns (mode name, {mode: [ms per step, ...]} or None, next frame)."""
    if choice != "auto":
        set_mode(INGEST_MODES[choice])
        return choice, None, f
    ms = {m: [] for m in INGEST_MODES}
    for _ in range(CAL_ROUNDS):
        for name, mode in INGEST_MODES.items():
            set_mode(mode)
            run_step(f)
            f += 1
            sync()
            t0 = time.perf_counter()
            for _ in range(CAL_STEPS):
                run_step(f)
                f += 1
            sync()
            ms[name].append((time.perf_counter() - t0) * 1e3 / CAL_STEPS)
    best = pick_ingest(ms)
    set_mode(INGEST_MODES[best])
    return best, {k: [round(x, 3) for x in v] for k, v in ms.items()}, f


PERIOD_S = 4.0                      # period of the synthetic trajectories: one rendered period is replayed for ever
REST_FRAMES = 6                     # frames 0..5 of a base stream show the platform at rest (gravity initialisation)
PERIOD_FRAMES = int(round(PERIOD_S / 0.04))
REST_IMU, PERIOD_IMU = 40, int(round(PERIOD_S / 0.005))
STAGGER = 3                         # start delay [frames] between sequences that replay the same base stream


def _render_base(args):
    """One base stream: REST_FRAMES frames at rest + one period of a periodic trajectory (xivo_b200.sim.periodic_trajectory), its IMU
    samples (rest: REST_IMU samples, then one period).  The trajectory returns to rest pose / zero velocity after a period, so the
    period can be replayed indefinitely as a physically consistent stream."""
    cfg, seed, channels = args
    from xivo_b200 import sim

    traj = sim.periodic_trajectory(PERIOD_S, amp_scale=0.85 + 0.1 * (seed % 4))
    msgs, _ = sim.image_stream(cfg, duration=0.2 + PERIOD_S + 0.04 + 1e-9, seed=seed, channels=channels, fast=True, traj=traj, rest_accel_is_gravity=True)
    frames = np.stack([p for k, _, p in msgs if k == "img"][: REST_FRAMES + PERIOD_FRAMES])
    imu = [p for k, _, p in msgs if k == "imu"][: REST_IMU + PERIOD_IMU]
    return frames, np.array([p[0] for p in imu]), np.array([p[1] for p in imu])


def make_base_streams(cfg, n_base, channels, procs):
    """Rendered before CUDA is initialised (fork pool)."""
    import multiprocessing as mp

    args = [(cfg, s, channels) for s in range(n_base)]
    if procs <= 1 or n_base == 1:
        return [_render_base(a) for a in args]
    with mp.get_context("fork").Pool(min(procs, n_base)) as pool:
        return pool.map(_render_base, args, chunksize=1)


def stream_tables(n_seq, n_base, n_frames, first_seq=0):
    """Which base-stream frame / IMU sample sequence s consumes at step f.  Sequence s replays base (s % n_base) after a start delay of
    (s // n_base) * STAGGER frames spent at rest, so at any step all sequences of a GPU read different frames (and sit in different
    phases of their state machines).  Returns (frame index (n_frames, n_seq), imu index (n_frames * 8, n_seq), base (n_seq,))."""
    s = np.arange(first_seq, first_seq + n_seq)
    base, delay = s % n_base, (s // n_base) * STAGGER
    f = np.arange(n_frames)[:, None]
    k = f - (REST_FRAMES - 1) - delay[None, :]          # motion phase in frames (k <= 0: still at rest)
    fidx = np.where(k <= 0, f % REST_FRAMES, REST_FRAMES - 1 + ((k - 1) % PERIOD_FRAMES) + 1)
    j = np.arange(n_frames * IMU_PER_FRAME)[:, None]
    jj = j - IMU_PER_FRAME * delay[None, :]
    iidx = np.where(jj < REST_IMU, j % REST_IMU, REST_IMU + ((jj - REST_IMU) % PERIOD_IMU))
    return fidx, iidx, base


def cpu_budget():
    """CPUs this process may use: affinity mask capped by the cgroup CPU quota (the GPU boxes run with one)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(q / p)))
        except Exception:
            pass
    return n


def parse_cpulist(text):
    out = []
    for tok in text.strip().split(","):
        if not tok:
            continue
        a, _, b = tok.partition("-")
        out.extend(range(int(a), int(b or a) + 1))
    return out


def pin_to_gpu_numa_node(local, lws):
    """Narrow this process to the CPUs of the NUMA node its GPU hangs off (pinned frame pool, table blobs and the library's host threads
    then sit next to the GPU's PCIe root) and tell the library which of the ranks of THAT node this one is (XIVO_CPU_SLICE), so that the
    ranks of a node split its cores without overlap.  No-op where sysfs has no NUMA information."""
    try:
        import torch

        def node_of(i):
            try:
                p = torch.cuda.get_device_properties(i)
                addr = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
            except AttributeError:  # older property set: ask NVML (same enumeration when CUDA_VISIBLE_DEVICES is unset)
                import pynvml

                pynvml.nvmlInit()
                bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(i)).busId
                bus = bus.decode() if isinstance(bus, bytes) else bus
                addr = bus.lower()[-12:]
            return int(open(f"/sys/bus/pci/devices/{addr}/numa_node").read())

        nodes = [node_of(i) for i in range(max(lws, local + 1))]
        me = nodes[local]
        if me < 0:
            return None
        allowed = os.sched_getaffinity(0)
        cpus = sorted(set(parse_cpulist(open(f"/sys/devices/system/node/node{me}/cpulist").read())) & allowed)
        peers = [i for i in range(lws) if nodes[i] == me] or [local]
        if len(cpus) < 2 * len(peers):
            return None
        os.sched_setaffinity(0, cpus)
        os.environ["XIVO_CPU_SLICE"] = f"{peers.index(local)}/{len(peers)}"
        return dict(node=me, cpus=len(cpus), rank_in_node=peers.index(local), ranks_in_node=len(peers))
    except Exception as e:  # noqa: BLE001 - placement is an optimisation, never a reason to fail
        log("numa placement skipped:", repr(e))
        return None


def cgroup_cpu_stat():
    """nr_throttled / throttled_usec / usage_usec of this container's CPU controller (cgroup v2), or None."""
    try:
        kv = dict(line.split() for line in open("/sys/fs/cgroup/cpu.stat"))
        return {k: int(kv[k]) for k in ("usage_usec", "nr_periods", "nr_throttled", "throttled_usec") if k in kv}
    except Exception:
        return None


def cpu_stat_delta(a, b, wall_ms):
    """CPU time the whole container used during a timed pass (in CPUs) and how much of the pass the quota throttled it."""
    if not a or not b:
        return None
    d = {k: b[k] - a[k] for k in a if k in b}
    return dict(cpus_used=round(d.get("usage_usec", 0) / (wall_ms * 1e3), 2), throttled_periods=d.get("nr_throttled"), periods=d.get("nr_periods"),
                throttled_ms=round(d.get("throttled_usec", 0) / 1e3, 1))


def cpu_baseline_entry(r, cores, frames, wall_s):
    """`cpu_baseline` object from oracle/cpu_baseline.py's result.  kind "reference": a frame costs the OpenCV tracker calls (cv2 LK + FAST
    on the image stream) plus the reference's OWN estimator (oracle/_ref/libxivo_ref_*.so, its unmodified sources) on a point-cloud
    stream of the same state size and track count; kind "port" (library absent): only the third-party numerics are timed (upper bound)."""
    upd_us = None
    if r.get("stage_share", {}).get("update") is not None and r.get("mean_frame_ms"):
        upd_us = r["stage_share"]["update"] * r["mean_frame_ms"] * 1e3  # Eigen 3.3.9 Joseph update (UpdateJosephForm's expression sequence), one core
        upd_us = round(upd_us, 2) if math.isfinite(upd_us) else None
    if r.get("fps_reference"):
        return dict(value=r["fps_reference"], ekf_update_us_per_frame=upd_us, unit="frames/s", cores=cores, kind="reference",
                    sample=(f"{cores} concurrent processes x {frames} frames: per frame cv2 LK+FAST on a synthetic 640x480 sequence ({r['tracker_ms']:.2f} ms) + the reference's own "
                            f"estimator library (propagation, ProcessTracks, sub-filters, Jacobians, gating, Joseph update, management) on a point-cloud stream with "
                            f"{r['ref_tracks']:.0f} tracks, state dim 89 ({r['ref_estimator_ms']:.2f} ms); {wall_s:.0f}s wall"),
                    numerics_only_value=r["fps"], numerics_only_note="cv2 LK+FAST + Eigen 3.3.9 gate/update only (kind port): upper bound on the reference", stage_share=r["stage_share"])
    return dict(value=r["fps"], ekf_update_us_per_frame=upd_us, unit="frames/s", cores=cores, kind="port",
                sample=f"{cores} concurrent synthetic 640x480 sequences x {frames} frames; timed: cv2 LK+FAST and Eigen-3.3.9 gate+update on the restated pipeline's inputs ({r['mean_frame_ms']:.2f} ms/frame/core, eigen={r['eigen']}, {wall_s:.0f}s)",
                stage_share=r["stage_share"])


def build_roofline(prof, K, peaks, seqs_per_launch, pass_ms):
    """Pure post-processing of the library's profile report (xivo_profile_report): per-kernel CUDA-event time and the
    algorithmic work attributed at the launch sites -> the `roofline` object of the JSON line (dominant kernel by device
    time; `achieved` = work per launch / average launch duration) and the host phase breakdown.  Unit-tested on CPU."""
    kern = {k: v for k, v in prof.items() if not k.startswith("_") and not k.startswith("host:")}
    host_phases = {k[5:]: round(v["ms"] / K, 4) for k, v in prof.items() if k.startswith("host:")}
    upd_ms = kern.get("ekf_gain", {}).get("ms", 0) + kern.get("ekf_cov", {}).get("ms", 0)
    merged = {k: dict(v) for k, v in kern.items() if k not in ("ekf_gain", "ekf_cov", "ekf_update")}
    if upd_ms:
        merged["ekf_update"] = dict(calls=kern.get("ekf_gain", {}).get("calls", 0), ms=upd_ms, work=kern.get("ekf_update", {}).get("work", 0))
    if not merged:
        return dict(kernel=None, bound=None, achieved=None, peak=None, unit=None, frac=None, traffic=None, kernels={}), host_phases
    tot_ms = sum(v["ms"] for v in merged.values()) or 1.0
    dom = max(merged, key=lambda k: merged[k]["ms"])
    d = merged[dom]
    bound = "tensor" if dom == "ekf_update" else "hbm"
    per_launch_s = max(d["ms"], 1e-9) * 1e-3 / max(d["calls"], 1)
    work_per_launch = d.get("work", 0) / max(d["calls"], 1)
    if bound == "hbm":
        achieved, peak, unit = work_per_launch / per_launch_s / 1e9, peaks["hbm"], "GB/s"
    else:
        achieved, peak, unit = work_per_launch / per_launch_s / 1e12, peaks["tf"], "TFLOP/s"
    traffic, traffic_src = None, None
    try:  # ncu-measured DRAM bytes per launch of that kernel (profiles/), scaled to this run's sequences per launch
        tname = "r02_traffic.json"
        tj = json.load(open(os.path.join(ROOT, "profiles", tname)))
        if dom in tj:
            traffic = tj[dom] * (seqs_per_launch / tj["sequences_per_launch"])
            traffic_src = "ncu dram__bytes_{read,write}.sum at %d sequences/launch (profiles/%s), scaled to %d" % (tj["sequences_per_launch"], tname, seqs_per_launch)
    except Exception:
        pass
    per_kernel = {}
    for k_, v_ in merged.items():  # the same arithmetic for every kernel with algorithmic work attributed (SURVEY.md §8d, csrc/estimator.cu add_work sites)
        if not v_.get("work") or not v_["ms"]:
            continue
        tens = k_ == "ekf_update"
        a_ = v_["work"] / (v_["ms"] * 1e-3) / (1e12 if tens else 1e9)
        per_kernel[k_] = dict(bound="tensor" if tens else "hbm", achieved=round(a_, 4), unit="TFLOP/s" if tens else "GB/s",
                              frac=round(a_ / (peaks["tf"] if tens else peaks["hbm"]), 6))
    # BASELINE.json's second headline figure: EKF measurement-update time per frame (gain + covariance kernels, one launch = one update of
    # every filter of a batch)
    upd = merged.get("ekf_update")
    ekf_update = None
    if upd and upd["calls"]:
        ekf_update = dict(us_per_frame=round(upd["ms"] * 1e3 / (upd["calls"] * seqs_per_launch), 4), us_per_launch=round(upd["ms"] * 1e3 / upd["calls"], 3),
                          filters_per_launch=seqs_per_launch, launches=upd["calls"], kernels="ekf_gain_kernel + ekf_cov_kernel (or ekf_cov_tc_kernel)")
    roofline = dict(kernel=dom, bound=bound, achieved=achieved, peak=peak, unit=unit, frac=achieved / peak, traffic=traffic, traffic_source=traffic_src, peak_source=peaks["src"],
                    per_kernel=per_kernel, ekf_update=ekf_update,
                    share_of_device_time=d["ms"] / tot_ms, launches=d["calls"], avg_launch_us=per_launch_s * 1e6,
                    kernels={k: dict(ms=round(v["ms"], 4), calls=v["calls"], share=round(v["ms"] / tot_ms, 4)) for k, v in merged.items()},
                    device_busy_frac=tot_ms / pass_ms, profiled_pass_ms_per_step=pass_ms / K,
                    attribution="third pass, batches stepped one after another (event durations = kernels, not queueing behind other batches)")
    return roofline, host_phases


DUMP_P_SEQS = 32  # covariances in a --dump-outputs directory: a fixed sample of sequences keeps it far below 64 MB at every config


def dump_outputs(out_dir, bts, sizes):
    """Writes what a caller of xivo_batch_step holds after the last step, for every sequence of this GPU in sequence order, as
    out_dir/<name>.npy (float64): the pose gsb, velocity, IMU biases and gravity rotation, the estimator counters, the tracked features
    (ids and pixel positions padded with -1: every value is finite) and the full error-state covariance of a seeded sample of the sequences."""
    seqs = [(b, s) for b, n in zip(bts, sizes) for s in range(n)]
    out = dict(gsb=np.stack([b.gsb(s) for b, s in seqs]))
    motion = [b.motion(s) for b, s in seqs]
    for i, name in enumerate(("vsb", "bg", "ba", "Rsg")):
        out[name] = np.stack([m[i] for m in motion])
    out["counters"] = np.array([list(b.counters(s).values()) for b, s in seqs], dtype=np.float64)
    tracked = [b.tracked_features(s)[:2] for b, s in seqs]
    width = max([len(ids) for ids, _ in tracked] + [1])
    out["tracked_ids"], out["tracked_xy"] = np.full((len(seqs), width), -1.0), np.full((len(seqs), width, 2), -1.0)
    for i, (ids, xy) in enumerate(tracked):
        out["tracked_ids"][i, : len(ids)], out["tracked_xy"][i, : len(ids)] = ids, xy
    pick = np.sort(np.random.default_rng(0).choice(len(seqs), min(DUMP_P_SEQS, len(seqs)), replace=False))
    out["P_sample_seqs"] = pick.astype(np.float64)
    out["P_sample"] = np.stack([seqs[i][0].P(seqs[i][1]) for i in pick])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name: a.shape for name, a in out.items()}


def run_ours(args):
    # host CPUs: the library's worker pool (workpool.h) is shared by the NB batches of this process; each batch
    # also has one driver thread (the Python thread inside xivo_batch_step), so workers + drivers = CPU budget
    lws = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    budget_all = cpu_budget()
    budget = max(1, budget_all // lws)
    # one driver per batch needs a CPU of its own: with a small budget (e.g. a node quota shared by 8 ranks) run fewer batches
    # a batch needs a driver thread; at least a quarter of the CPUs stay with the workers.  (Half, the rule until r02ae, turned the 12 CPUs a
    # rank gets on a multi-GPU box into 6 batches of 171 sequences: two waves of the CTA-per-filter kernels on 148 SMs.)
    args.batches = max(1, min(args.batches, budget * 3 // 4))
    os.environ.setdefault("XIVO_THREADS", str(max(1, min(args.max_threads, budget) - args.batches + 1 - args.cpu_headroom)))
    os.environ.setdefault("XIVO_DRIVERS", str(args.batches))
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # every lane has its own streams: more hardware queues than the default 8, fewer false dependencies
    os.environ.setdefault("XIVO_PIN_DRIVERS", "1")  # the batch driver threads are ours: let the library pin them next to its workers
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    cfg = load_cfg()
    cfg["covariance_update"] = args.cov_update  # "fp64" (default, exact parity) or "tf32x3" (tcgen05 downdate, fp32 accuracy)
    B, K, W, FPS, CH = args.seqs, args.steps, args.warmup, args.frames_per_step, args.channels
    S0 = max(1, min(args.streams, B))
    # ---- synthetic inputs (rendered before CUDA is initialised: fork pool) ----
    t0 = time.time()
    bases = make_base_streams(cfg, S0, CH, max(1, budget - 1))
    log(f"rendered {S0} base streams x {REST_FRAMES + PERIOD_FRAMES} frames in {time.time() - t0:.1f}s")
    import torch

    from xivo_b200 import capi, pyxivo, replicas

    torch.cuda.set_device(local)
    numa = pin_to_gpu_numa_node(local, lws) if args.numa else None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    NFB = REST_FRAMES + PERIOD_FRAMES
    fshape = (ROWS, COLS) if CH == 1 else (ROWS, COLS, CH)
    fbytes = ROWS * COLS * CH
    host = torch.empty((S0, NFB) + fshape, dtype=torch.uint8).pin_memory()  # the pool every step reads from (e2e pass)
    for s, (frames, _, _) in enumerate(bases):
        host[s] = torch.from_numpy(frames)
    dev = host.cuda()                                                          # the same pool resident in HBM (device-resident pass)
    base_g = np.stack([b[1] for b in bases])  # (S0, REST_IMU + PERIOD_IMU, 3)
    base_a = np.stack([b[2] for b in bases])
    del bases
    # ---- schedule: which frame / IMU sample every sequence consumes at every step ----
    K_prof = min(K, args.profile_steps)
    n_cal = calibration_frames(args.ingest)
    max_delay = ((world * B - 1) // S0) * STAGGER
    PREROLL = max_delay + 20  # every sequence has left its rest phase, initialised gravity and vision, and filled its state
    n_total = PREROLL + FPS * (2 * (W + K) + (W + K_prof)) + n_cal + 8 + (64 if args.single_stream else 0)
    fidx, iidx, base = stream_tables(B, S0, n_total, first_seq=rank * B)
    frame_ts = (np.arange(n_total, dtype=np.uint64) * np.uint64(FRAME_NS))
    imu_ts_all = (np.arange(n_total * IMU_PER_FRAME, dtype=np.uint64) * np.uint64(FRAME_NS // IMU_PER_FRAME))

    NB = max(1, min(args.batches, B))
    sizes = [B // NB + (1 if i < B % NB else 0) for i in range(NB)]
    L = capi.lib()
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor

    L.xivo_ctx_stream.restype = C.c_void_p
    ctxs, bts, exts, tabs = [], [], [], []
    o = 0
    for nb in sizes:
        c = capi.Context(local)
        ctxs.append(c)
        bts.append(pyxivo.Batch(cfg, n_seq=nb, max_groups=G, max_features=F, ctx=c))
        exts.append(torch.cuda.ExternalStream(L.xivo_ctx_stream(c._h)))
        sl = slice(o, o + nb)
        # everything a step passes to the C ABI is laid out once, so that the timed loop is the C call and nothing else
        t = dict(its=np.ascontiguousarray(np.broadcast_to(imu_ts_all[:, None], (n_total * IMU_PER_FRAME, nb))),
                 ig=np.ascontiguousarray(base_g[base[sl][None, :], iidx[:, sl]]),   # (n_total * 8, nb, 3)
                 ia=np.ascontiguousarray(base_a[base[sl][None, :], iidx[:, sl]]),
                 fts=np.ascontiguousarray(np.broadcast_to(frame_ts[:, None], (n_total, nb))),
                 hptr=np.ascontiguousarray(np.uint64(host.data_ptr()) + (base[sl][None, :].astype(np.uint64) * np.uint64(NFB) + fidx[:, sl].astype(np.uint64)) * np.uint64(fbytes)),
                 dptr=np.ascontiguousarray(np.uint64(dev.data_ptr()) + (base[sl][None, :].astype(np.uint64) * np.uint64(NFB) + fidx[:, sl].astype(np.uint64)) * np.uint64(fbytes)))
        t["addr"] = {k: v.ctypes.data for k, v in t.items()}
        t["row"] = {k: v.strides[0] for k, v in t.items() if k != "addr"}
        tabs.append(t)
        o += nb
    pool = ThreadPoolExecutor(NB)
    VP = C.c_void_p
    pending = [-1] * NB  # per batch: the frame whose upload xivo_batch_prefetch_frames has started

    def step_one(i, f, device_resident):
        t = tabs[i]
        ad, rw = t["addr"], t["row"]
        j = f * IMU_PER_FRAME
        stream = not device_resident and args.prefetch

        def prefetch_next():
            # streaming ingest: the copy of frame f + 1 overlaps the computation of frame f and is consumed by the next call; every step
            # still uploads exactly one frame per sequence inside the timed region
            if L.xivo_batch_prefetch_frames(bts[i]._h, VP(ad["hptr"] + (f + 1) * rw["hptr"]), ROWS, COLS, CH) != 0:
                raise RuntimeError(L.xivo_last_error().decode())
            pending[i] = f + 1

        primed = stream and pending[i] == f  # frame f is already on its way (prefetched by the previous call)
        if primed:
            prefetch_next()
        else:
            pending[i] = -1  # whatever was pending is dropped by the library: these are other buffers
        rc = L.xivo_batch_step(bts[i]._h, IMU_PER_FRAME, VP(ad["its"] + j * rw["its"]), VP(ad["ig"] + j * rw["ig"]), VP(ad["ia"] + j * rw["ia"]),
                               VP(ad["fts"] + f * rw["fts"]), VP((ad["dptr"] if device_resident else ad["hptr"]) + f * rw["hptr"]), ROWS, COLS, CH, int(device_resident))
        if rc != 0:
            raise RuntimeError(L.xivo_last_error().decode())
        if stream and not primed:
            prefetch_next()
        return bts[i].gsb(0)  # host read of the step's result (pose); the err/P_mm D2H happened inside the call

    def frame_step(f, device_resident, serial=False):
        if NB == 1 or serial:
            return [step_one(i, f, device_resident) for i in range(NB)]
        return list(pool.map(lambda i: step_one(i, f, device_resident), range(NB)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
            torch.cuda.synchronize()

    f = 0
    for _ in range(PREROLL):
        frame_step(f, True)
        f += 1
    log("preroll done", PREROLL, "frames;", bts[0].counters(0), bts[-1].counters(sizes[-1] - 1))

    def timed(device_resident, profile, K_):
        """W warm-up steps, then exactly K_ timed steps; one step = FPS consecutive frames (+ their IMU samples) of every sequence."""
        nonlocal f
        for _ in range(W * FPS):
            frame_step(f, device_resident)
            f += 1
        L.xivo_profile_reset()
        L.xivo_profile_enable(int(profile))
        launches0 = capi.launch_count()
        clk = ClockSampler(local)
        barrier()
        cst0 = cgroup_cpu_stat()
        clk.start()
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(NB)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(NB)]
        t0 = time.perf_counter()
        for i in range(NB):
            e0[i].record(exts[i])
        ntracked = 0
        for _ in range(K_ * FPS):
            # the attribution pass steps the batches one after another: with several batches in flight a CUDA-event pair
            # around a launch also measures the time the launch queued behind other batches' kernels
            frame_step(f, device_resident, serial=bool(profile) and not args.profile_overlapped)
            f += 1
        ntracked = float(np.mean([bts[i].counters(s)["num_tracked"] for i in range(NB) for s in range(0, sizes[i], max(1, sizes[i] // 8))]))
        for i in range(NB):
            e1[i].record(exts[i])
        barrier()
        wall = time.perf_counter() - t0
        cst = cpu_stat_delta(cst0, cgroup_cpu_stat(), wall * 1e3)
        clocks = clk.stop()
        ms = max(e0[0].elapsed_time(e1[i]) for i in range(NB))  # first start -> last end, on the launch streams
        L.xivo_profile_enable(0)
        buf = C.create_string_buffer(1 << 16)
        L.xivo_profile_report(buf, len(buf))
        prof = json.loads(buf.value.decode())
        ms = replicas.max_over_ranks(ms, device="cuda")
        return dict(ms=ms, wall_ms=wall * 1e3, prof=prof, launches=capi.launch_count() - launches0, clocks=clocks, ntracked=ntracked, cpu_stat=cst)

    # three passes over consecutive frames of the same streams: the two measured ones run with the in-library
    # profiler off (its event records and locks cost ~1 ms/step); the third only attributes time to kernels
    r_dev = timed(True, 0, K)
    log("device-resident pass", r_dev["ms"], "ms")
    L.xivo_set_frame_ingest.restype = C.c_int

    def cal_step(k):
        frame_step(k, False)

    ingest, ingest_cal, f = calibrate_ingest(args.ingest, L.xivo_set_frame_ingest, cal_step, torch.cuda.synchronize, f)
    log("frame ingest:", ingest, ingest_cal)
    r_e2e = timed(False, 0, K)
    log("e2e pass", r_e2e["ms"], "ms")
    r_prof = timed(not args.profile_e2e, args.profile_level, K_prof)
    log("profiled pass", r_prof["ms"], "ms")
    if args.dump_outputs and rank == 0:
        log("outputs written to", args.dump_outputs, dump_outputs(args.dump_outputs, bts, sizes))
    frames_total = world * B * K * FPS
    value = frames_total / (r_dev["ms"] * 1e-3)
    e2e = frames_total / (r_e2e["ms"] * 1e-3)

    # single-sequence latency (BASELINE.md: the reference runs ONE stream at 1-7 ms per frame): a batch of one, host frames, synchronous
    single = None
    if args.single_stream and rank == 0:
        b1 = pyxivo.Batch(cfg, n_seq=1, max_groups=G, max_features=F, ctx=ctxs[0])
        t1 = tabs[0]
        lat = []
        for ff in range(48):
            j = ff * IMU_PER_FRAME
            its = np.ascontiguousarray(t1["its"][j : j + IMU_PER_FRAME, :1])
            ig = np.ascontiguousarray(t1["ig"][j : j + IMU_PER_FRAME, :1])
            ia = np.ascontiguousarray(t1["ia"][j : j + IMU_PER_FRAME, :1])
            fts = np.ascontiguousarray(t1["fts"][ff, :1])
            ptr = (C.c_void_p * 1)(int(t1["hptr"][ff, 0]))
            tq = time.perf_counter()
            rc = L.xivo_batch_step(b1._h, IMU_PER_FRAME, VP(its.ctypes.data), VP(ig.ctypes.data), VP(ia.ctypes.data), VP(fts.ctypes.data), ptr, ROWS, COLS, CH, 0)
            b1.gsb(0)
            lat.append((time.perf_counter() - tq) * 1e3)
            if rc != 0:
                raise RuntimeError(L.xivo_last_error().decode())
        lat = np.array(lat[24:])  # frames after the reorder buffer filled and the first detections happened
        single = dict(ms_per_frame_median=float(np.median(lat)), ms_per_frame_p95=float(np.percentile(lat, 95)), fps=float(1e3 / np.median(lat)),
                      note="one sequence, batch of 1, host frame in -> pose out per call (wall clock); the reference's published single-stream figure is 140 FPS (BASELINE.md)")
        b1.close()

    peaks = measured_peaks()
    roofline, host_phases = build_roofline(r_prof["prof"], K_prof * FPS, peaks, sizes[0], r_prof["ms"])

    out = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            # CPUs the cgroup quota lets us run concurrently (measured before the library pinned this thread: pin_driver narrows the affinity mask)
            cores = min(budget_all, args.cpu_cores) if args.cpu_cores else budget_all
            t0 = time.time()
            log("cpu baseline on", cores, "cores")
            r = cpu_reference(cores, 60, 14, CH)
            cpu = cpu_baseline_entry(r, cores, 60, time.time() - t0)
        pool_mb = S0 * NFB * fbytes / 1e6
        out = dict(metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=K, warmup=W,
                   ms_per_step=r_dev["ms"] / K, higher_is_better=True, scaling="weak", vs_baseline=None,
                   dtype="f64" if args.cov_update == "fp64" else "f64 state, 3xTF32 tensor-core covariance downdate", data="synthetic",
                   config=dict(covariance_update=args.cov_update, workload=WORKLOAD,
                               sequences_per_gpu=B, batches_per_gpu=NB, lanes_per_batch=bts[0].lanes, cpu_tokens=os.environ.get("XIVO_CPU_TOKENS"), frames_per_sequence_per_step=FPS, frames_per_step=world * B * FPS,
                               host_threads=int(os.environ.get("XIVO_THREADS", "0")) or None, host_cpu_budget=budget, channels=CH,
                               distinct_streams=f"{S0} base streams (own texture / trajectory amplitude / noise, period {PERIOD_S:g} s replayed) x start delays of {STAGGER} frames: "
                                                f"no two sequences of a GPU read the same frame in the same step",
                               l2_policy=f"inputs larger than L2: a step reads {B * FPS} distinct frames ({B * FPS * fbytes / 1e6:.0f} MB) per GPU out of a {pool_mb:.0f} MB frame pool; "
                                         f"covariances and pyramids are the resident state by design",
                               message_buffer_size=cfg.get("message_buffer_size", 10), frame_ingest=ingest, frame_prefetch=bool(args.prefetch), numa=numa,
                               frame_ingest_calibration_ms_per_step=ingest_cal),
                   e2e=dict(value=e2e, unit="frames/s", h2d_bytes_per_step=r_e2e["prof"]["_h2d_bytes"] / K if r_e2e["prof"]["_h2d_bytes"] else world * B * FPS * fbytes,
                            d2h_bytes_per_step=(r_e2e["prof"]["_d2h_bytes"] / K) if r_e2e["prof"]["_d2h_bytes"] else None, ms_per_step=r_e2e["ms"] / K),
                   gpu_launches=r_dev["launches"], clocks=r_dev["clocks"], roofline=roofline, cpu_baseline=cpu, single_stream=single,
                   tracked_features_mean=r_dev["ntracked"], wall_ms_per_step=r_dev["wall_ms"] / K, host_phase_ms_per_frame_step=host_phases,
                   host_cpu=dict(value_pass=r_dev["cpu_stat"], e2e_pass=r_e2e["cpu_stat"], note="container CPU time / wall of the pass and cgroup quota throttling (cpu.stat), rank 0's view of the whole container"))
        print(json.dumps(out))
    pool.shutdown()
    for b_ in bts:
        b_.close()
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()
    return out


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the same path on this box's host cores (oracle/cpu_baseline.py: cv2 tracker
    calls + the reference's own estimator library built from its unmodified sources), one sequence per allowed CPU.  A step is the
    same unit as in the CUDA arm (--frames-per-step consecutive frames of every sequence), on a bounded sample: at most 240 timed
    frames per sequence, so that the run ends within a few minutes whatever K the driver asks for."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = min(cpu_budget(), args.cpu_cores) if args.cpu_cores else cpu_budget()  # CPUs the cgroup quota lets us run concurrently
    K, W, FPS = args.steps, args.warmup, args.frames_per_step
    frames = min(K * FPS, 240)
    t0 = time.time()
    r = cpu_reference(cores, frames, PREROLL_FRAMES + min(W * FPS, 24), args.channels)
    cb = cpu_baseline_entry(r, cores, frames, time.time() - t0)
    ms_per_step = 1e3 * cores * FPS / cb["value"]  # one step = FPS frames on each of `cores` concurrent sequences
    out = dict(impl="reference", metric=METRIC, value=cb["value"], unit="frames/s", n_gpus=args.gpus,
               steps=K, warmup=W, ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
               config=dict(workload=WORKLOAD,
                           sequences=cores, frames_per_sequence_per_step=FPS, timed_frames_per_sequence=frames, channels=args.channels),
               cpu_baseline=cb,
               e2e=dict(value=cb["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cpu-headroom", type=int, default=1, help="CPUs of the quota left to Python / CUDA helper threads")
    ap.add_argument("--profile-e2e", action="store_true", help="attribute kernel / host-phase time on the host-frame (e2e) path instead of the device-resident one")
    ap.add_argument("--profile-level", type=int, default=1, help="1: kernels + batch-level host phases, 2: + per-sequence host scopes")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(CONFIGS), help="BASELINE.json configs[n]: 1 = the headline workload (640x480, 150 features, N=89); 2 = TUM-VI equidistant 512x512, 200 features, N=203; 3 = stress 1280x1024, 800 features, N=299")
    ap.add_argument("--seqs", type=int, default=0, help="independent sequences per GPU, split over --batches lock-step batches (0 = the config's default: 1024 / 256 / 128)")
    ap.add_argument("--batches", type=int, default=8, help="separate lock-step xivo_batch handles per GPU, each stepped from its own thread; their per-sequence host code shares the library's worker pool (capped at half the CPU budget)")
    ap.add_argument("--streams", type=int, default=0, help="rendered base streams (texture / trajectory / noise); every sequence replays one of them with its own start delay")
    ap.add_argument("--frames-per-step", type=int, default=8, help="a step = this many consecutive frames (+ IMU) of every sequence: K driver-chosen steps then time seconds, not milliseconds")
    ap.add_argument("--channels", type=int, default=1, choices=[1, 3], help="1 = grey frames (default), 3 = BGR like the reference's cv::imread input (src/app/vio.cpp:72)")
    ap.add_argument("--profile-steps", type=int, default=4, help="steps of the (serial, slow) kernel-attribution pass")
    ap.add_argument("--profile-overlapped", action="store_true", help="attribution pass with the batches in flight together (event durations then include queueing)")
    ap.add_argument("--max-threads", type=int, default=16, help="cap on host threads per rank (workers + drivers): more than this measured slower (SCALE_r01: 88 threads 2.3x slower than 16)")
    ap.add_argument("--no-single-stream", dest="single_stream", action="store_false", help="skip the batch-of-one latency measurement")
    ap.add_argument("--cpu-cores", type=int, default=0)
    ap.add_argument("--cov-update", default="fp64", choices=["fp64", "tf32x3"], help="arithmetic of the covariance downdate (tf32x3 = tcgen05 tensor cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa", dest="numa", action="store_false", help="leave the process on every allowed CPU instead of the NUMA node of its GPU")
    ap.add_argument("--prefetch", action="store_true", help="e2e pass with xivo_batch_prefetch_frames (the upload of frame k + 1 is started before frame k is processed); measured neutral on the B200 box (profiles/r02z_sweep.txt), so the default is the plain call")
    ap.add_argument("--ingest", default="auto", choices=["auto"] + list(INGEST_MODES), help="how pinned host frames reach the device (e2e pass); auto = calibrate both before the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed passes, write the state every sequence of GPU 0 holds after its last step "
                                                          "(pose, motion, counters, tracked features, a seeded sample of covariances) as DIR/<name>.npy; "
                                                          "the inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repository's path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3
    c = select_config(args.config)
    args.seqs = args.seqs or c["seqs"]
    args.streams = args.streams or c["streams"]
    if args.impl == "reference" and args.config == 3:
        # the reference's estimator is a compile-time-sized build (EKF_MAX_GROUPS / EKF_MAX_FEATURES); oracle/build_ref.py builds G4_F14 and G15_F30
        print(json.dumps(dict(impl="reference", unavailable="reference estimator not built for G=15,F=62 (configs[3]); configs 1 and 2 are")))
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
