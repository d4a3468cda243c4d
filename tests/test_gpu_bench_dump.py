"""bench.py --dump-outputs: the files hold the system the timed path assembled, so that two builds can be compared on them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.common import rel_frobenius
from tests.gpu_common import run_product

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_timed_system(tmp_path):
    """At a small mesh every entry is written (no sampling): the dump equals one IGAComputeSystem of the same workload."""
    from bench import build_case
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--mesh", "12", "--steps", "2", "--no-cpu-baseline", "--no-configs",
                        "--no-solve", "--no-e2e", "--no-quad", "--no-parity", "--dump-outputs", str(out)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    d = {name[:-len(".npy")]: np.load(out / name) for name in os.listdir(out)}
    assert set(d) == {"matrix_values", "matrix_rows", "matrix_cols", "rhs", "rhs_index"}
    assert all(a.dtype == np.float64 for a in d.values())
    res = run_product(build_case(12), "SYSTEM", "POISSON", path="auto")
    rp = res["rowptr"]
    assert np.array_equal(d["matrix_rows"], np.repeat(np.arange(len(rp) - 1), np.diff(rp)))
    assert np.array_equal(d["matrix_cols"], res["colidx"])
    assert np.array_equal(d["rhs_index"], np.arange(len(res["rhs"])))
    assert rel_frobenius(d["matrix_values"], res["values"]) <= 1e-12 and rel_frobenius(d["rhs"], res["rhs"]) <= 1e-12
