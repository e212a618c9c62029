"""Host logic of the estimator on CPU (no GPU, no nvcc): tests/cpp/host_harness.cpp compiles the product's host
state machine (xivo_b200/csrc/estimator.h + estimator_host.cpp.inc) with g++ and exposes the pieces that need no
kernel output — configuration, message heap, clocks, gravity initialisation, the nominal-state Runge-Kutta chain with
the per-stage records the device covariance kernel consumes, and the tracker mask — which are checked here against
the numpy oracle (oracle/estimator_oracle.py, oracle/ekf_oracle.py, oracle/tracker_oracle.py)."""
import ctypes as C
import heapq
import json
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import ekf_oracle as E
from oracle import estimator_oracle as EO
from oracle import tracker_oracle as T
from xivo_b200 import sim

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = os.path.join(ROOT, "xivo_b200", "cfg")
CUDA_INC = os.environ.get("CUDA_HOME", "/usr/local/cuda") + "/include"
pytestmark = pytest.mark.skipif(shutil.which("g++") is None or not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")),
                                reason="needs g++ and the CUDA headers (host-only compile)")


@pytest.fixture(scope="module")
def hh(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hh") / "libhost_harness.so")
    cmd = ["g++", "-std=c++17", "-O2", "-march=x86-64-v3", "-I", CUDA_INC, "-shared", "-fPIC", os.path.join(ROOT, "tests", "cpp", "host_harness.cpp"), "-o", so]
    if os.environ.get("XIVO_HH_SO"):  # a pre-built harness, e.g. one compiled with -fsanitize=address,undefined (run under LD_PRELOAD=libasan.so)
        so = os.environ["XIVO_HH_SO"]
    else:
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    lib.hh_create.restype = C.c_void_p
    lib.hh_create.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int]
    lib.hh_error.restype = C.c_char_p
    lib.hh_curr_time.restype = C.c_ulonglong
    for name in ("hh_destroy", "hh_motion", "hh_flags", "hh_initial_pmm", "hh_camera", "hh_mask_reset", "hh_mask_dump"):
        getattr(lib, name).argtypes = [C.c_void_p] + ([C.c_void_p] if name not in ("hh_destroy", "hh_mask_reset") else [])
    lib.hh_curr_time.argtypes = [C.c_void_p]
    lib.hh_sticky_error.argtypes = [C.c_void_p]
    lib.hh_inertial.argtypes = [C.c_void_p, C.c_ulonglong, C.c_void_p, C.c_void_p]
    lib.hh_visual_begin.argtypes = [C.c_void_p, C.c_ulonglong, C.c_int]
    lib.hh_take_stages.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.hh_push.argtypes = [C.c_void_p, C.c_ulonglong, C.c_int]
    lib.hh_pop.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.hh_mask_init.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.hh_triangulate.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p]
    lib.hh_mask_out.argtypes = [C.c_void_p, C.c_double, C.c_double]
    lib.hh_mask_valid.argtypes = [C.c_void_p, C.c_double, C.c_double]
    return lib


def create(lib, cfg, G=4, F=14, tracker_only=False):
    text = cfg if isinstance(cfg, str) else json.dumps(cfg)
    h = lib.hh_create(text.encode(), G, F, int(tracker_only))
    return h


def motion(lib, h):
    a = np.zeros(42)
    lib.hh_motion(h, a.ctypes.data)
    return dict(Rsb=a[:9].reshape(3, 3), Tsb=a[9:12], Vsb=a[12:15], bg=a[15:18], ba=a[18:21], Rbc=a[21:30].reshape(3, 3), Tbc=a[30:33], Rsg=a[33:42].reshape(3, 3))


def take_stages(lib, h):
    buf = np.zeros((1024, 16))
    n = lib.hh_take_stages(h, buf.ctypes.data, 1024)
    return buf[:n].copy()


# ------------------------------------------------------------------ configuration
def test_config_files_parse_with_comments_and_camera_models(hh):
    for name, model, rows in [("pcw_sim.json", 0, 480), ("vio_640x480.json", 0, 480), ("tumvi_512_equidistant.json", 3, 512), ("stress_1280x1024.json", 0, 1024)]:
        text = open(os.path.join(CFG, name)).read()
        assert "//" in text  # the files carry comments, like the reference's cfg/*.json
        h = create(hh, text)
        assert h, hh.hh_error()
        cam = np.zeros(11)
        hh.hh_camera(h, cam.ctypes.data)
        ref = sim.load_cfg(os.path.join(CFG, name))["camera_cfg"]
        assert int(cam[0]) == model and int(cam[1]) == rows and cam[3] == ref["fx"] and cam[6] == ref["cy"]
        if model == 3:
            assert np.array_equal(cam[7:11], ref["k0123"])
        hh.hh_destroy(h)


@pytest.mark.parametrize("key,value,needle", [("use_OOS", True, "MSCKF"),
                                               ("integration_method", "Euler", "integration method"), ("covariance_update", "fp16", "covariance_update")])
def test_unsupported_options_fail_loudly_at_creation(hh, key, value, needle):
    cfg = sim.load_cfg(os.path.join(CFG, "pcw_sim.json"))
    cfg[key] = value
    assert not create(hh, cfg)
    assert needle.lower() in hh.hh_error().decode().lower()


def test_unsupported_camera_model_is_an_error(hh):
    cfg = sim.load_cfg(os.path.join(CFG, "pcw_sim.json"))
    cfg["camera_cfg"]["model"] = "radtan"
    assert not create(hh, cfg) and b"radtan" in hh.hh_error()


def test_initial_motion_covariance_matches_oracle(hh):
    cfg = sim.load_cfg(os.path.join(CFG, "vio_640x480.json"))
    h = create(hh, cfg)
    P = np.zeros((23, 23))
    hh.hh_initial_pmm(h, P.ctypes.data)
    ref = EO.EstimatorOracle(cfg, G=4, F=14)
    assert np.array_equal(P, ref.P[:23, :23])  # estimator.cpp:258-302
    m = motion(hh, h)
    assert np.allclose(m["Rbc"], ref.X.Rbc, atol=1e-15) and np.array_equal(m["Tbc"], ref.X.Tbc)
    hh.hh_destroy(h)


# ------------------------------------------------------------------ message heap
def test_message_heap_order_matches_the_reference_rule(hh):
    """MaintainBuffer (estimator.cpp:923-941): nothing executes until more than MESSAGE_BUFFER_SIZE (10) messages are held;
    then the front of a std heap ordered by timestamp ONLY pops, so ties resolve the way libstdc++'s heap algorithms do.
    The product's host code and the oracle's helper (oracle/stdumap.cpp) must replay exactly the same sequence."""
    from oracle import stdorder as SO

    h = create(hh, sim.load_cfg(os.path.join(CFG, "pcw_sim.json")))
    rng = np.random.default_rng(0)
    ts = rng.integers(0, 40, 400) * 5_000_000  # many ties
    types = rng.integers(0, 2, 400) * 3
    ref = SO.StdMessageHeap(10)
    popped_ref, popped = [], []
    for k in range(400):
        hh.hh_push(h, int(ts[k]), int(types[k]))
        due = ref.push(int(ts[k]), (int(ts[k]), int(types[k])))
        t, ty = C.c_ulonglong(), C.c_int()
        got = hh.hh_pop(h, C.byref(t), C.byref(ty))
        assert got == (1 if due is not None else 0) == (1 if k >= 10 else 0)
        if got:
            popped.append((t.value, ty.value))
            popped_ref.append(due)
    assert popped == popped_ref and len(popped) == 390  # the last 10 messages are never executed, as in the reference
    # timestamps come out non-decreasing once the stream itself is (almost) ordered
    ordered = sorted(int(x) for x in ts)
    h2 = create(hh, sim.load_cfg(os.path.join(CFG, "pcw_sim.json")))
    out = []
    for x in ordered:
        hh.hh_push(h2, x, 0)
        t, ty = C.c_ulonglong(), C.c_int()
        if hh.hh_pop(h2, C.byref(t), C.byref(ty)):
            out.append(t.value)
    assert out == ordered[:390]
    hh.hh_destroy(h)
    hh.hh_destroy(h2)


# ------------------------------------------------------------------ inertial path
@pytest.mark.parametrize("method", ["PrinceDormand", "RK4"])
def test_nominal_state_chain_and_stage_records_match_oracle(hh, method, monkeypatch):
    cfg = sim.load_cfg(os.path.join(CFG, "pcw_sim.json"))
    cfg["integration_method"] = method
    msgs, _ = sim.pcw_stream(cfg, duration=0.5, seed=3)
    h = create(hh, cfg)
    ref = EO.EstimatorOracle(cfg, G=4, F=14)
    rec = []
    real = E.integrate
    monkeypatch.setattr(EO.E, "integrate", lambda *a, **k: real(*a, rec=rec, **k))
    nst = 7 if method == "PrinceDormand" else 4
    n_imu = n_vis = 0
    for kind, ts, p in msgs:
        if kind == "imu":
            g, a = np.ascontiguousarray(p[0]), np.ascontiguousarray(p[1])
            hh.hh_inertial(h, ts, g.ctypes.data, a.ctypes.data)
            ref.inertial_internal(ts, g, a)
            n_imu += 1
        else:  # the clock / propagate part of a visual message (estimator.cpp:1106-1122); the update itself needs the device
            assert hh.hh_visual_begin(h, ts, 3) == (1 if ref.gravity_initialized else 0)
            if not ref.vision_initialized:
                if ref.gravity_initialized:
                    ref.curr_time, ref.vision_initialized = ts, True
            else:
                ref.last_time, ref.curr_time = ref.curr_time, ts
            if ref.vision_initialized:
                ref.propagate(True)
            n_vis += 1
        got = take_stages(hh, h)
        assert len(got) == len(rec) and len(got) % nst == 0
        if len(rec):
            want = np.array(rec)
            assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max())
            assert np.array_equal(np.sign(got[:, 15]), np.sign(want[:, 15]))  # the sign of h marks the end of a Propagate call
        rec.clear()
        m = motion(hh, h)
        assert np.abs(m["Rsb"] - ref.X.Rsb).max() <= 1e-12 and np.abs(m["Tsb"] - ref.X.Tsb).max() <= 1e-12
        assert np.abs(m["Vsb"] - ref.X.Vsb).max() <= 1e-12 and np.abs(m["Rsg"] - ref.X.Rsg).max() <= 1e-15
        assert hh.hh_curr_time(h) == ref.curr_time
    assert n_imu == 100 and n_vis >= 12 and np.linalg.norm(ref.X.Tsb) > 0.05  # it moved
    fl = (C.c_int * 4)()
    hh.hh_flags(h, fl)
    assert list(fl) == [1, 1, ref.imu_counter, n_vis]
    hh.hh_destroy(h)


def test_out_of_order_messages_are_dropped_and_wrong_mode_is_sticky(hh):
    cfg = sim.load_cfg(os.path.join(CFG, "pcw_sim.json"))
    h = create(hh, cfg)
    z, a = np.zeros(3), np.array([0.0, 0.0, 9.8])
    hh.hh_inertial(h, 0, z.ctypes.data, a.ctypes.data)
    assert hh.hh_visual_begin(h, 40_000_000, 3) == 1
    hh.hh_inertial(h, 45_000_000, z.ctypes.data, a.ctypes.data)
    n0 = len(take_stages(hh, h))
    assert n0 > 0
    hh.hh_inertial(h, 20_000_000, z.ctypes.data, a.ctypes.data)  # older than the clock (ms granularity): dropped, estimator.cpp:706-717
    assert len(take_stages(hh, h)) == 0 and hh.hh_curr_time(h) == 45_000_000
    assert hh.hh_visual_begin(h, 30_000_000, 3) == 0 and hh.hh_sticky_error(h) == 0
    assert hh.hh_visual_begin(h, 80_000_000, 1) == 0 and hh.hh_sticky_error(h) == -3  # VisualMeas in simulation mode (estimator.cpp:1112-1115)
    hh.hh_destroy(h)


def test_gravity_initialisation_from_stationary_samples(hh):
    cfg = sim.load_cfg(os.path.join(CFG, "vio_640x480.json"))  # simulation: false, gravity_init_counter: 20
    h = create(hh, cfg)
    ref = EO.EstimatorOracle(cfg, G=4, F=14)
    rng = np.random.default_rng(4)
    tilt = E.so3_exp(np.array([0.05, -0.08, 0.3]))
    for k in range(25):
        g = rng.normal(0, 1e-3, 3)
        a = tilt @ np.array([0.0, 0.0, 9.8]) + rng.normal(0, 1e-2, 3)
        hh.hh_inertial(h, k * 5_000_000, g.ctypes.data, a.ctypes.data)
        ref.inertial_internal(k * 5_000_000, g, a)
        fl = (C.c_int * 4)()
        hh.hh_flags(h, fl)
        assert bool(fl[0]) == ref.gravity_initialized == (k >= 19)
    m = motion(hh, h)
    assert np.abs(m["Rsg"] - ref.X.Rsg).max() <= 1e-14 and not np.allclose(m["Rsg"], np.eye(3), atol=1e-3)
    w = E.so3_log(m["Rsg"]) if hasattr(E, "so3_log") else None
    assert w is None or abs(w[2]) < 1e-12  # the yaw component of Wsg is dropped (estimator.cpp:461)
    hh.hh_destroy(h)


# ------------------------------------------------------------------ tracker mask
@pytest.mark.parametrize("rows,cols", [(480, 640), (67, 130), (64, 64)])
def test_tracker_mask_matches_oracle(hh, rows, cols):
    cfg = sim.load_cfg(os.path.join(CFG, "vio_640x480.json"))
    h = create(hh, cfg)
    tcfg = cfg["tracker_cfg"]
    ref = T.Mask(rows, cols, tcfg["margin"], tcfg["mask_size"])
    ref.reset()
    hh.hh_mask_init(h, rows, cols)
    out = np.zeros((rows, cols), np.uint8)
    hh.hh_mask_dump(h, out.ctypes.data)
    assert np.array_equal(out, ref.m)
    rng = np.random.default_rng(rows)
    for k in range(max(8, rows * cols // 1500)):
        x, y = rng.uniform(-10, cols + 10), rng.uniform(-10, rows + 10)
        if k % 7 == 0:
            x, y = np.floor(x) + 0.5, np.floor(y) + 0.5  # cvRound ties (half to even)
        assert bool(hh.hh_mask_valid(h, x, y)) == ref.valid(x, y)
        hh.hh_mask_out(h, x, y)
        ref.mask_out(x, y)
    hh.hh_mask_dump(h, out.ctypes.data)
    assert np.array_equal(out, ref.m) and 0 < (out > 0).sum() < rows * cols
    hh.hh_mask_reset(h)
    ref.reset()
    hh.hh_mask_dump(h, out.ctypes.data)
    assert np.array_equal(out, ref.m)
    hh.hh_destroy(h)


# ------------------------------------------------------------------------------------------------------------------------
# Two-view triangulation (csrc/triangulate.h) against the restatement of helpers.cpp:103-372 in oracle/ekf_oracle.py
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mi,method", list(enumerate(E.TRI_METHODS)))
def test_triangulation_matches_the_oracle(hh, mi, method):
    rng = np.random.default_rng(100 + mi)
    n_ok = n_bad = 0
    for trial in range(400):
        # a point in front of view 0, view 1 displaced by a small motion, pixel-noise-like perturbation of both rays
        X0 = np.array([rng.uniform(-2, 2), rng.uniform(-2, 2), rng.uniform(0.5, 12.0)])
        R01 = E.so3_exp(rng.normal(0, 0.05, 3))
        t01 = rng.normal(0, 0.3, 3)
        X1 = R01.T @ (X0 - t01)
        if X1[2] < 0.2:
            continue
        xc0 = X0[:2] / X0[2] + rng.normal(0, 0.004 if trial % 3 else 0.0002, 2)
        xc1 = X1[:2] / X1[2] + rng.normal(0, 0.004 if trial % 3 else 0.0002, 2)
        zmin, zmax = 0.05, (5.0 if trial % 2 else 60.0)
        th, beta = math.radians(0.1 if trial % 4 else 2.0), math.radians(0.25)
        want = E.triangulate(method, R01, t01, xc0, xc1, zmin, zmax, th, beta)
        out = np.zeros(3)
        ok = hh.hh_triangulate(mi, np.ascontiguousarray(R01).ctypes.data, t01.ctypes.data, np.ascontiguousarray(xc0).ctypes.data,
                               np.ascontiguousarray(xc1).ctypes.data, C.c_double(zmin), C.c_double(zmax), C.c_double(th), C.c_double(beta), out.ctypes.data)
        assert bool(ok) == (want is not None), f"{method} trial {trial}: acceptance differs"
        if ok:
            n_ok += 1
            # rounding is amplified by 1 / sin(parallax) in the angular forms (and by the singular-value gap in L2); the DLT variants solve ill-conditioned systems at small parallax (error ~ eps / sin^2(parallax))
            tol = 1e-10 if "angular" in method else 1e-7
            assert np.abs(out - want).max() <= tol * max(1.0, np.abs(want).max()), f"{method} trial {trial}: {out} vs {want}"
        else:
            n_bad += 1
    assert n_ok >= 40 and n_bad >= 10, (n_ok, n_bad)


def test_triangulation_config_is_parsed_like_the_reference(hh):
    """estimator.cpp:157-164, :356-358: method default l1_angular, degrees -> radians, a wrong method is fatal (feature.cpp:724-728)."""
    cfg = sim.load_cfg(os.path.join(CFG, "pcw_sim.json"))
    cfg.update({"triangulate_pre_subfilter": True, "triangulation": {"method": "no_such_method"}})
    assert not hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0) and b"Triangulation" in hh.hh_error()
    cfg["triangulation"] = {"zmax": 60.0}
    h = hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0)
    assert h, hh.hh_error()
    hh.hh_destroy(h)


def test_host_triangulation_on_the_reference_known_answers(hh):
    """src/test/unittest_triangulation.cpp:18-206 through csrc/triangulate.h (fixtures shared with tests/test_oracle_ekf.py)."""
    import test_oracle_ekf as TO

    for name, xc1, z1, g21, noise, expect in TO.reference_triangulation_fixtures():
        R12, t12, x1, x2 = TO.reference_triangulation_inputs(xc1, z1, g21, noise)
        for mi in (2, 3, 4):  # l1, l2, linf
            out = np.zeros(3)
            ok = hh.hh_triangulate(mi, np.ascontiguousarray(R12).ctypes.data, t12.ctypes.data, x1.ctypes.data, x2.ctypes.data, C.c_double(0.0),
                                   C.c_double(1e9), C.c_double(0.1 * math.pi / 180), C.c_double(0.25 * math.pi / 180), out.ctypes.data)
            assert bool(ok) == expect, f"{name}: {E.TRI_METHODS[mi]}"
            if expect:
                assert abs(math.exp(out[2]) - z1) <= 0.5


def test_tracker_only_accepts_the_reference_tracker_only_config_shape(hh):
    """CreateSystemTrackerOnly (factory.cpp:84-122) is fed configs with only camera_cfg (model, rows, cols) + tracker_cfg
    (cfg/tumvi_tracker_only_cam0.json); the full estimator still insists on its filter sections."""
    full = sim.load_cfg(os.path.join(CFG, "vio_640x480.json"))
    cfg = {"simulation": False, "print_timing": False, "use_canvas": True, "async_run": False,
           "camera_cfg": {"model": "equidistant", "rows": 512, "cols": 512}, "tracker_cfg": dict(full["tracker_cfg"])}
    h = hh.hh_create(json.dumps(cfg).encode(), 15, 30, 1)
    assert h, hh.hh_error()
    hh.hh_destroy(h)
    assert not hh.hh_create(json.dumps(cfg).encode(), 15, 30, 0)  # not a valid estimator config


def test_descriptor_options_follow_the_reference_constructor(hh):
    """Tracker::Tracker (tracker.cpp:176-217): the rescue of dropped tracks needs descriptors (LOG(FATAL) "must extract descriptors in order
    to match dropped tracks"), the MATCH tracker too; a distance threshold switches the extraction on; only BRIEF is built."""
    cfg = sim.load_cfg(os.path.join(CFG, "vio_640x480.json"))
    cfg["tracker_cfg"]["match_dropped_tracks"] = True
    assert not hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0) and b"must extract descriptors" in hh.hh_error()
    cfg["tracker_cfg"]["extract_descriptor"] = True
    h = hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0)
    assert h, hh.hh_error()
    hh.hh_destroy(h)
    cfg["tracker_cfg"].update(extract_descriptor=False, match_dropped_tracks=False, tracker_type="MATCH")
    assert not hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0) and b"matcher-tracker requires" in hh.hh_error()
    cfg["tracker_cfg"].update(descriptor_distance_thresh=50)  # > -1 implies extraction (tracker.cpp:178-179)
    h = hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0)
    assert h, hh.hh_error()
    hh.hh_destroy(h)
    cfg["tracker_cfg"].update(descriptor="ORB")
    assert not hh.hh_create(json.dumps(cfg).encode(), 4, 14, 0) and b"ORB" in hh.hh_error()


# ------------------------------------------------------------------------------------------------------------------------
# Tracker-level outlier rejection (csrc/homography.h): cv::findHomography's inlier mask, LMEDS and RANSAC
# ------------------------------------------------------------------------------------------------------------------------
def _homography_scene(rng, structured):
    n = int(rng.integers(12, 160))  # (below ~8 points LMedS's median falls inside the exact-fit sample: its "best" model is decided by 1e-10 float noise)
    p0 = rng.uniform(8, 630, (n, 2)).astype(np.float32)
    if not structured:  # unrelated point sets: every hypothesis has its own inlier set -> pins the cv::RNG draws and checkSubset
        return p0, rng.uniform(8, 630, (n, 2)).astype(np.float32), 3.0
    H0 = np.eye(3) + rng.normal(0, [[0.01, 0.01, 3], [0.01, 0.01, 3], [1e-5, 1e-5, 0]])
    q = np.c_[p0, np.ones(n)] @ H0.T
    p1 = (q[:, :2] / q[:, 2:]).astype(np.float32) + rng.normal(0, rng.choice([0.3, 1.0, 2.0]), (n, 2)).astype(np.float32)
    k = int(n * rng.uniform(0, 0.4))
    p1[:k] += rng.normal(0, 30, (k, 2)).astype(np.float32)
    return p0, p1.astype(np.float32), float(rng.choice([1.5, 3.0, 4.0]))


@pytest.mark.parametrize("method", [4, 8], ids=["LMEDS", "RANSAC"])
def test_homography_mask_matches_the_oracle_and_cv2(hh, method):
    from oracle import homography_oracle as HO

    try:
        import cv2
    except ImportError:
        cv2 = None
    hh.hh_homography_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, C.c_void_p]
    rng = np.random.default_rng(40 + method)
    flips = 0
    for trial in range(48):
        p0, p1, thr = _homography_scene(rng, structured=trial % 4 != 0)
        n = len(p0)
        ok, want, _H = HO.find_homography_mask_413(p0, p1, method, thr, 2000, 0.995)
        got = np.zeros(n, np.uint8)
        rc = hh.hh_homography_mask(p0.ctypes.data, p1.ctypes.data, n, method, C.c_double(thr), 2000, C.c_double(0.995), got.ctypes.data)
        assert bool(rc) == ok
        # the threshold test on the refined model is the only place where 1e-7 of difference in H (Jacobi eigenvectors vs LAPACK,
        # Gaussian elimination vs eigen-solve) can flip a point that sits exactly on the threshold
        flips += int((got != want).sum())
        if cv2 is not None and trial % 4 != 0:  # (on unrelated point sets the LM refinement runs on a meaningless fit; cv2's solver and ours part at 1e-3 there)
            _Hc, mc = cv2.findHomography(p0, p1, method, thr, maxIters=2000, confidence=0.995)
            flips += int((got != (np.zeros(n, np.uint8) if mc is None else mc.ravel())).sum())
    assert flips <= 2, f"{flips} mask entries differ over 48 scenes"


# the configs shipped in the reference's cfg/ directory, parsed (tests/golden/make_golden_cfgs.py)
REFERENCE_CFGS = os.path.join(ROOT, "tests", "golden", "reference_cfgs.json")
# what each estimator / tracker config shipped with the reference does when it is handed to the host parser unmodified
# (None = accepted; otherwise a fragment of the refusal).  DESIGN.md §8 discusses every entry.
SHIPPED = {
    "pcw.json": None, "pcw_loops.json": None, "phab.json": None, "tumvi_cam1.json": None,
    "tumvi_cam0.json": None,                # the reference's flagship config: BRIEF descriptors + rescue of dropped tracks (match_dropped_tracks)
    "void_params.json": "Wsb",              # stale in the reference itself: state keys W / T / V (its use_1pt_RANSAC is accepted: Estimator::OnePointRANSAC is built)
    "phab_calibration.json": "json",        # stale in the reference itself: `"method": 1`, state keys W / T / V
    "void_params_calib.json": "Wsb",        # stale in the reference itself: state keys W / T / V
    "tumvi_tracker_only_cam0.json": None, "tumvi_tracker_only_cam1.json": None,  # (LMEDS outlier rejection + descriptor rescue on)
    "phab_tracker_only.json": "SIFT",       # MATCH tracker is built, its SIFT descriptor is not (BRIEF only)
    "void_tracker_only.json": "radtan",
}


@pytest.mark.parametrize("name,refusal", sorted(SHIPPED.items()))
def test_shipped_reference_configs_through_the_host_parser(hh, name, refusal):
    with open(REFERENCE_CFGS) as f:
        cfg = json.load(f)[name]
    h = hh.hh_create(json.dumps(cfg).encode(), 15, 30, int("tracker_only" in name))
    if refusal is None:
        assert h, hh.hh_error()
        hh.hh_destroy(h)
    else:
        assert not h and refusal.lower() in hh.hh_error().decode().lower(), hh.hh_error()
    if name == "phab_tracker_only.json":  # with BRIEF in place of SIFT the shipped MATCH-tracker file runs as it is
        cfg["tracker_cfg"]["descriptor"] = "BRIEF"
        h = hh.hh_create(json.dumps(cfg).encode(), 15, 30, 1)
        assert h, hh.hh_error()
        hh.hh_destroy(h)
