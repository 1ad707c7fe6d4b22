"""The reference arm of bench.py (baseline/ref_arm.py) runs the UNMODIFIED reference from baseline/_ref/solver, which
__graft_entry__.build() installs where a checkout of the reference is available.  These CPU tests pin it: BASELINE config 1
(20^3 Kuhn cube Poisson, CG to 1e-8) through the reference's own `stable_conjugate_gradient_solver` gives the 133 iterations /
u_max 0.50102 that SURVEY.md section 6 probed, and agrees with the numpy oracle on the same problem.  Without the reference,
the oracle is compared with the reference's stored output (tests/golden/reference_config1.json)."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import GOLDEN, PKG, ROOT

ARM = os.path.join(ROOT, "baseline", "ref_arm.py")
HAVE_REF = os.path.exists(os.path.join(ROOT, "baseline", "_ref", "solver", "solver.py"))


def test_reference_arm_config1_and_oracle():
    c1 = json.load(open(os.path.join(GOLDEN, "reference_config1.json")))
    if HAVE_REF:
        r = subprocess.run([sys.executable, ARM, "--n", "6", "--iters", "3", "--c1"], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = r.stdout.strip().splitlines()
        assert len(lines) == 1, "the arm prints exactly one JSON line (the reference's own prints are captured)"
        d = json.loads(lines[0])
        assert d["tets"] == 6 * 6 ** 3 and d["iters"] == 3 and d["rate"] > 0
        assert d["c1"]["iterations"] == c1["iterations"] and abs(d["c1"]["u_max"] - c1["u_max"]) < 1e-8
        c1 = d["c1"]
    assert c1["iterations"] == 133 and abs(c1["u_max"] - 0.50102) < 1e-4
    # the numpy oracle on the same problem: same iteration count, same maximum
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    from femb200 import meshgen
    from oracle import fem_oracle as O
    c, t = meshgen.kuhn_cube(20)
    c, t = c.numpy(), t.numpy()
    Ke = O.c3d4_poisson_K(c, t)
    load = np.bincount(t.reshape(-1), weights=np.repeat(O.tet_volumes(c, t) / 4, 4), minlength=c.shape[0]).reshape(-1, 1)
    u, it, st = O.stable_cg(Ke, t, load, np.flatnonzero(c[:, 2] == 0), tol=1e-8, ndof=1)
    assert st == "converged" and abs(it - c1["iterations"]) <= 1 and abs(float(u.max()) - c1["u_max"]) < 1e-8


def test_reference_arm_never_loads_the_product():
    """The arm must stay free of the product (its `native_so_loaded` is checked by the driver): no femb200 / libfemb200 import."""
    src = open(ARM).read()
    assert "import femb200" not in src and "from femb200" not in src and "libfemb200" not in src.replace("never imports femb200 / libfemb200.so", "")


def test_bench_reference_line_shape():
    """`bench.py --impl reference` prints ONE JSON line with the contract's keys, kind = reference when the reference is installed,
    otherwise the C port of the same loop, labelled as such."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3", "--cpu-n", "10"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["metric"] == "cg_iters_per_s" and d["value"] > 0
    if HAVE_REF:
        assert d["cpu_baseline"]["kind"] == "reference" and "NOT extrapolated" in d["cpu_baseline"]["sample"]
    else:
        assert d["cpu_baseline"]["kind"] == "port" and "not extrapolated" in d["cpu_baseline"]["sample"] and "NOT the reference" in d["note"]
