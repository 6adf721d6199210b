"""The bounded select of the affinity graph (group minima from the distance GEMM, one filtered pass
over the row) against the bound-free selects it replaces, bit for bit, on the rows the predecessor
pin does not reach: candidates overflowing the per-row buffer (1200 equal feature rows), graphs with
exactly k and k + 1 valid nodes (rows without a bound take the exact fallback), and n = 6544, the
ScanNet-shape 3-way graph.  The bound-free reference is the measurement build with the register-fed
distance GEMM (R3DFS_DIST_TC=1), which writes no group minima and gives the same distances."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,case", [(4416, "dup"), (4416, "exact_k"), (6544, "base")])
def test_bounded_select_equals_bound_free_select(n, case, tmp_path):
    script = os.path.join(os.path.dirname(os.path.dirname(__file__)), "scripts", "check_select.py")
    a, b = str(tmp_path / "a.pt"), str(tmp_path / "b.pt")
    from r3dfsseg_b200 import _lib
    assert os.path.isfile(_lib.AB_LIB_PATH), "measurement build missing: make -C r3dfsseg_b200/csrc ab"
    env_old = dict(os.environ, R3DFS_LIB=_lib.AB_LIB_PATH, R3DFS_DIST_TC="1")
    subprocess.run([sys.executable, script, "run", a, str(n), "3", case], check=True, timeout=300)
    subprocess.run([sys.executable, script, "run", b, str(n), "3", case], check=True, timeout=300,
                   env=env_old)
    r = subprocess.run([sys.executable, script, "cmp", a, b], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
