"""Generates tests/golden/reference_cfgs.json: the estimator / tracker configs shipped with the reference (its cfg/ directory), each
parsed the way xivo_b200.sim.load_cfg parses a file (comments stripped).  tests/test_host_logic.py hands every one of them to the
host parser unmodified and checks which are accepted and why the others are refused.

  python tests/golden/make_golden_cfgs.py <reference checkout>/cfg"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from test_host_logic import SHIPPED  # noqa: E402
from xivo_b200 import sim  # noqa: E402

cfg_dir = sys.argv[1]
out = {name: sim.load_cfg(os.path.join(cfg_dir, name)) for name in sorted(SHIPPED)}
with open(os.path.join(ROOT, "tests", "golden", "reference_cfgs.json"), "w") as f:
    json.dump(out, f, indent=1)
    f.write("\n")
print(len(out), "configs")
