"""Generates tests/golden/reference_pcw.npz by running the REFERENCE'S OWN ESTIMATOR (oracle/_ref/libxivo_ref_*.so, built from the
unmodified sources under /root/reference by oracle/build_ref.py) on the point-cloud streams of tests/test_reference_pin.py.  Only
possible where the reference library is built (the authoring container).  The arrays pin the oracle and, through it, the CUDA pipeline."""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref_runner  # noqa: E402
from test_reference_pin import CASES, CFG  # noqa: E402

out = {}
with tempfile.TemporaryDirectory() as td:
    for name, G, F, duration, seed, sim_depths, over, offset in CASES:
        d = ref_runner.run_subprocess(CFG, G, F, duration, seed, sim_depths, os.path.join(td, name + ".npz"), overrides=over, pc_offset_ns=offset)
        for k in ("gsb", "ts", "n_instate", "gauge", "ids"):
            out[f"{name}.{k}"] = d[k]
        out[f"{name}.P_upper"] = d["P"][np.triu_indices(len(d["P"]))]  # symmetric to 1e-19 (test_reference_pin.sym_from_upper)
        if name in ("small_89", "default_203"):  # the reference's read-back accessors at the end of the run (boundary-parity fixtures)
            for k in d.files:
                if k.startswith("acc."):
                    out[f"{name}.{k}"] = d[k]
        print(name, d["gsb"].shape, int(d["n_instate"][-1]), np.round(d["gsb"][-1][:, 3] - d["truth"][-1], 4))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "reference_pcw.npz"), **out)
