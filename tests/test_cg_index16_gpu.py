"""The merged CG loop streams a 16-bit delta-encoded column index (DESIGN 3.4) when the operator allows it.  Every case is
compared bit for bit (u, rs, iteration count) with the same solve on the int32 kernel, forced by FEMB_SPMV_IDX32=1 in a
subprocess, and `info["index_bytes"]` shows which index the loop streamed.  The operators have at most 592 row tiles of 128
rows, so both kernels run one CTA per tile and their per-CTA partial sums match; on larger operators the two kernels' CTA
counts differ (5 against 4 per SM) and the dot products are summed in a different order."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import PKG, ROOT

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(PKG, "solver"))
DEV = "cuda:0"
FEW = (3, 4000)  # couplings 70,000 apart: 4 of the 586 tiles of a 75,000-row chain escape (< 1 %)


def _chain(n, far_pairs=(), far=70_000, headless_row=None):
    """SPD chain operator (4 on the diagonal, -1 to both neighbours) plus symmetric couplings -0.5 between i and i + far for
    i in far_pairs: those rows' gaps exceed 65535, so their tiles escape to the int32 path.  headless_row: a row whose
    diagonal and left neighbour are dropped (first column above the row); the mask holds it at zero."""
    rows = {i: {i: 4.0} for i in range(n)}
    for i in range(n - 1):
        rows[i][i + 1] = rows[i + 1][i] = -1.0
    for i in far_pairs:
        rows[i][i + far] = rows[i + far][i] = -0.5
    if headless_row is not None:
        del rows[headless_row][headless_row], rows[headless_row][headless_row - 1]
    crow, col, val = [0], [], []
    for i in range(n):
        for c in sorted(rows[i]):
            col.append(c), val.append(rows[i][c])
        crow.append(len(col))
    return np.array(crow, np.int32), np.array(col, np.int32), np.array(val)


def _ring(n, stride):
    """Periodic chain with neighbours i +- stride: three entries in every row, the same row pointers for every stride."""
    crow = np.arange(0, 3 * n + 1, 3, dtype=np.int32)
    col = np.sort(np.stack([(np.arange(n) - stride) % n, np.arange(n), (np.arange(n) + stride) % n], 1), 1).astype(np.int32)
    val = np.where(col == np.arange(n)[:, None], 4.0, -1.0)
    return crow, col.reshape(-1), val.reshape(-1)


def _kuhn(n=30):
    import element as el
    from femb200 import meshgen
    c, t = meshgen.kuhn_cube(n, jitter=0.1)
    plan = el.CsrPlan(t, c.shape[0], DEV)
    crow, col = plan.pattern(1)
    vals = plan.assemble_c3d4(c, "poisson")
    mask = (c[:, 2] != 0).to(torch.uint8).to(DEV)
    F = torch.linspace(1.0, 2.0, c.shape[0], dtype=torch.float64).to(DEV)
    return crow, col, vals, F, mask


def _dev(crow, col, val):
    return torch.from_numpy(crow).to(DEV), torch.from_numpy(col).to(DEV), torch.from_numpy(val).to(DEV)


def run_cases():
    """Every case of this file: name -> (u, rs, iterations, index_bytes).  Run in-process and, with FEMB_SPMV_IDX32=1, in a
    subprocess."""
    from femb200 import ops
    out = {}

    def keep(name, u, info):
        out[name] = (u.detach().cpu().clone(), info["rs"], info["iterations"], info["index_bytes"])

    crow, col, vals, F, mask = _kuhn()
    for tol, it in ((0.0, 60), (1e-9, 2000)):
        keep(f"kuhn_cg_{tol}", *ops.cg_solve(crow, col, vals, F, mask=mask, tol=tol, max_iter=it))
        minv = ops.jacobi(crow, col, vals, mask)
        keep(f"kuhn_pcg_{tol}", *ops.cg_solve(crow, col, vals, F, mask=mask, minv=minv, tol=tol, max_iter=it))
    keep("kuhn_short", *ops.cg_solve(crow, col, vals, F, mask=mask, tol=0.0, max_iter=8))

    n = 75_000  # 586 tiles
    c, k, v = _dev(*_chain(n, far_pairs=FEW))
    Fc = torch.cos(torch.arange(n, dtype=torch.float64, device=DEV))
    keep("chain_few_escape", *ops.cg_solve(c, k, v, Fc, tol=0.0, max_iter=60))
    keep("chain_few_escape_tol", *ops.cg_solve(c, k, v, Fc, tol=1e-9, max_iter=2000))
    c, k, v = _dev(*_chain(n, far_pairs=range(0, n - 70_000, 50)))
    keep("chain_many_escape", *ops.cg_solve(c, k, v, Fc, tol=0.0, max_iter=60))
    c, k, v = _dev(*_chain(20_000, headless_row=1300))
    m = torch.ones(20_000, dtype=torch.uint8, device=DEV)
    m[1300] = 0
    keep("headless_row", *ops.cg_solve(c, k, v, Fc[:20_000], mask=m, tol=0.0, max_iter=60))

    # the column index changed in place between two calls with the same tensors: re-encoded, same as a fresh solve
    n = 40_000
    c, k, v = _dev(*_ring(n, 1))
    Fr = torch.sin(torch.arange(n, dtype=torch.float64, device=DEV))
    keep("ring_before", *ops.cg_solve(c, k, v, Fr, tol=0.0, max_iter=40))
    k.copy_(torch.from_numpy(_ring(n, 2)[1]).to(DEV))
    keep("ring_in_place", *ops.cg_solve(c, k, v, Fr, tol=0.0, max_iter=40))
    keep("ring_fresh", *ops.cg_solve(c.clone(), k.clone(), v.clone(), Fr.clone(), tol=0.0, max_iter=40))
    return out


@pytest.fixture(scope="module")
def results(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("idx32") / "idx32.pt")
    code = ("import sys, torch, importlib.util; sys.path[:0] = [{root!r}, {pkg!r}, {tests!r}]; "
            "spec = importlib.util.spec_from_file_location('idx16_cases', {me!r}); m = importlib.util.module_from_spec(spec); "
            "spec.loader.exec_module(m); torch.save(m.run_cases(), {path!r})").format(
                root=ROOT, pkg=PKG, tests=os.path.join(ROOT, "tests"), me=os.path.abspath(__file__), path=path)
    env = dict(os.environ, FEMB_SPMV_IDX32="1")
    subprocess.run([sys.executable, "-c", code], env=env, check=True, timeout=900)
    return run_cases(), torch.load(path)


def _same(a, b):
    return torch.equal(a[0], b[0]) and a[1] == b[1] and a[2] == b[2]


@pytest.mark.parametrize("name", ["kuhn_cg_0.0", "kuhn_cg_1e-09", "kuhn_pcg_0.0", "kuhn_pcg_1e-09", "chain_few_escape",
                                  "chain_few_escape_tol", "headless_row", "ring_before", "ring_in_place"])
def test_index16_bit_identical_to_int32(results, name):
    new, old = results
    assert new[name][3] == 2 and old[name][3] == 4, (name, new[name][3], old[name][3])
    assert _same(new[name], old[name]), (name, new[name][1:], old[name][1:])


def test_index16_converging_solves_converge(results):
    new, _ = results
    for name in ("kuhn_cg_1e-09", "kuhn_pcg_1e-09", "chain_few_escape_tol"):
        assert new[name][2] < 2000 and new[name][1] ** 0.5 < 1e-9, (name, new[name][1:])


def test_index16_short_solve_and_escaping_matrix_use_int32(results):
    new, old = results
    for name in ("kuhn_short", "chain_many_escape"):
        assert new[name][3] == 4 and _same(new[name], old[name]), (name, new[name][1:], old[name][1:])


def test_index16_in_place_column_change_matches_fresh_solve(results):
    new, _ = results
    assert _same(new["ring_in_place"], new["ring_fresh"])
    assert not torch.equal(new["ring_in_place"][0], new["ring_before"][0])


def test_index16_escaping_tiles_match_oracle(results):
    from oracle import c_oracle
    new, _ = results
    crow, col, val = _chain(75_000, far_pairs=FEW)
    F = np.cos(np.arange(75_000, dtype=np.float64))
    u, it, st = c_oracle.cg_csr(crow, col, val, F, np.zeros(0, np.int64), tol=1e-9, max_iter=2000)
    assert st == "converged" and abs(new["chain_few_escape_tol"][2] - it) <= 1
    assert np.abs(new["chain_few_escape_tol"][0].numpy() - u).max() <= 1e-8 * np.abs(u).max()
