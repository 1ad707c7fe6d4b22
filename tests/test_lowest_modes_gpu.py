"""lowest_modes on the GPU: each block kernel of csrc/modes.cu against its numpy restatement (oracle/modes_oracle.py), and the
public solver against dense / shift-invert references and against the numpy-backend driver."""
import os
import sys

import numpy as np
import pytest
import scipy.linalg as sl
import scipy.sparse.linalg as sla
import torch

from conftest import PKG

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(PKG, "solver"))

DEV = "cuda:0"
KW = dict(device=DEV, dtype=torch.float64)


@pytest.fixture(scope="module")
def env():
    import element
    import solver
    from femb200 import meshgen, modes, ops
    from oracle import modes_oracle as MO
    return element, solver, meshgen, modes, ops, MO


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def backends(env, coords, conn, Kloc, Mloc, fixed, n_nodes):
    """DeviceBackend and NumpyBackend on the same assembled K, M and mask."""
    el, sv, meshgen, modes, ops, MO = env
    dev = torch.device(DEV)
    plan = ops.cached_plan(conn, n_nodes, dev)
    brow, bcol = plan.pattern(1)
    K = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Kloc, 3))
    M = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Mloc, 3))
    mask = sv._dof_mask(n_nodes, 3, fixed, dev)
    dbe = modes.DeviceBackend(K, M, mask)
    nbe = MO.NumpyBackend(brow.cpu().numpy(), bcol.cpu().numpy(), K.bval.cpu().numpy(), M.bval.cpu().numpy(), mask.cpu().numpy())
    return dbe, nbe


def c3d4_case(env, n=4, fixed_face=True, isolated=False):
    el, sv, meshgen, *_ = env
    c, t = meshgen.kuhn_cube(n, jitter=0.2)
    N = c.shape[0] + (1 if isolated else 0)   # an extra node no element touches
    if isolated:
        c = torch.cat([c, torch.full((1, 3), 2.0, dtype=c.dtype)])
    K = el.compute_c3d4_K_matrix(c, t, 1.0, 0.3, **KW)
    M = el.compute_c3d4_M_matrix(c, t, 2.5, **KW)
    fixed = torch.nonzero(c[:, 0] == 0).reshape(-1) if fixed_face else torch.zeros(0, dtype=torch.int64)
    return c, t.to(DEV), K, M, fixed, N


def test_kernels_match_numpy_restatement(env):
    el, sv, meshgen, modes, ops, MO = env
    c, t, K, M, fixed, N = c3d4_case(env, n=5, isolated=True)
    dbe, nbe = backends(env, c, t, K, M, fixed, N)
    n = dbe.n
    rng = np.random.default_rng(7)
    # SpMM at m = 1, 4, 7, 16, with and without M and the mask (the isolated node gives an empty block row)
    for m in (1, 4, 7, 16):
        for with_m in (True, False):
            for masked in (True, False):
                ld = 3 * m + 1
                Xh = rng.standard_normal((n, ld))
                dmask, nmask = dbe.mask, nbe.mask
                if not masked:
                    dbe.mask, nbe.mask = None, np.ones(n, dtype=np.uint8)
                Yd = [dbe.zeros(n, ld), dbe.zeros(n, ld) if with_m else None]
                Yn = [np.zeros((n, ld)), np.zeros((n, ld)) if with_m else None]
                dbe.spmm(dbe.upload(Xh), 1, m, *Yd) if with_m else dbe_spmm_k_only(dbe, dbe.upload(Xh), 1, m, Yd[0])
                nbe.spmm(Xh, 1, m, *Yn)
                dbe.mask, nbe.mask = dmask, nmask
                assert rel(Yd[0].cpu().numpy()[:, 1:1 + m], Yn[0][:, 1:1 + m]) <= 1e-13, (m, with_m, masked)
                if with_m:
                    assert rel(Yd[1].cpu().numpy()[:, 1:1 + m], Yn[1][:, 1:1 + m]) <= 1e-13, (m, masked)
                assert float(Yd[0][-3:].abs().max()) == 0.0          # isolated node: y = 0
    # Gram at (1,1), (16,48), (48,48) with n not a multiple of the 32-row tile
    nr = 1000 * 32 + 17
    for ka, kb in ((1, 1), (16, 48), (48, 48)):
        A, B = rng.standard_normal((nr, 48)), rng.standard_normal((nr, 50))
        G = dbe.zeros(1, ka * kb).reshape(-1)
        from femb200._lib import check, lib
        Ad, Bd = dbe.upload(A), dbe.upload(B)          # held until the kernel has run
        check(lib.femb_mb_gram(nr, ka, modes._p(Ad), 48, kb, modes._p(Bd), 50, modes._p(G), dbe.stream))
        assert rel(G.cpu().numpy().reshape(ka, kb), A[:, :ka].T @ B[:, :kb]) <= 1e-13, (ka, kb)
    # combine with beta != 0 into an interleaved view
    X = rng.standard_normal((n, 48))
    Cm = rng.standard_normal((40, 12))
    Yh = rng.standard_normal((n, 16))
    Yd = dbe.upload(Yh)
    dbe.combine(dbe.upload(X), 40, Cm, Yd, 3, beta=-0.5)
    Yn = Yh.copy()
    nbe.combine(X, 40, Cm, Yn, 3, beta=-0.5)
    assert rel(Yd.cpu().numpy(), Yn) <= 1e-13
    # residual with locked columns: W gets the active ones, packed
    m = 12
    S = rng.standard_normal((n, 3 * m)) * nbe.mask[:, None]
    KS, MS = rng.standard_normal((n, 3 * m)), rng.standard_normal((n, 3 * m))
    lam = rng.standard_normal(m)
    active = [1, 4, 5, 9, 11]
    Sd, nd = dbe.upload(S), dbe.zeros(1, 2 * m).reshape(-1)
    dbe.residual(Sd, dbe.upload(KS), dbe.upload(MS), m, lam, dbe.active_list(active), len(active), Sd, m, nd)
    nn = np.zeros(2 * m)
    nbe.residual(S, KS, MS, m, lam, np.array(active), len(active), S, m, nn)
    assert rel(Sd.cpu().numpy(), S) <= 1e-13 and rel(nd.cpu().numpy(), nn) <= 1e-13


def dbe_spmm_k_only(dbe, X, c0, k, YK):
    from femb200._lib import check, lib
    from femb200 import modes
    K = dbe.K
    check(lib.femb_spmm_bsr3(K.nb, K.nnzb, modes._p(K.brow), modes._p(K.bcol), modes._p(K.bval), None, modes._p(dbe.mask), k,
                             modes._p(X, c0), X.shape[1], modes._p(YK, c0), None, YK.shape[1], dbe.stream), "femb_spmm_bsr3")


def dense_check(env, c, conn, K, M, fixed, N, num_eigs=6):
    el, sv, meshgen, modes, ops, MO = env
    lam, X, info = sv.lowest_modes(K, M, conn, fixed, N, num_eigs=num_eigs, tol=1e-10, max_iter=1000, return_info=True, verbose=False, **KW)
    assert info["status"] == "converged", info
    _, nbe = backends(env, c, conn, K, M, fixed, N)
    free = nbe.mask.astype(bool)
    Kd, Md = nbe.K.toarray()[np.ix_(free, free)], nbe.M.toarray()[np.ix_(free, free)]
    ex, V = sl.eigh(Kd, Md)
    from test_lowest_modes_cpu import assert_same_modes
    Xh = X.cpu().numpy()
    assert np.abs(Xh[~free]).max() == 0.0
    assert_same_modes(lam.cpu().numpy(), Xh[free], ex, V, Md, 1e-8, 1e-6)
    return lam, X, info


def test_lowest_modes_c3d4_c3d10_c3d8_match_dense(env):
    el, sv, meshgen, *_ = env
    c, t, K, M, fixed, N = c3d4_case(env)
    dense_check(env, c, t, K, M, fixed, N)
    c, t = meshgen.tet10_cube(2, jitter=0.1)
    fixed = torch.nonzero(c[:, 0] == 0).reshape(-1)
    dense_check(env, c, t.to(DEV), el.compute_c3d10_K_matrix(c, t, 1.0, 0.3, **KW), el.compute_c3d10_M_matrix(c, t, 2.5, **KW), fixed,
                c.shape[0])
    c, h = meshgen.hex_cube(4, jitter=0.1)
    fixed = torch.nonzero(c[:, 0] == 0).reshape(-1)
    dense_check(env, c, h.to(DEV), el.compute_c3d8_K_matrix(c, h, 1.0, 0.3, **KW), el.compute_c3d8_M_matrix(c, h, 2.5, **KW), fixed,
                c.shape[0], num_eigs=5)


def test_larger_cantilever_matches_shift_invert(env):
    el, sv, meshgen, modes, ops, MO = env
    c, t, K, M, fixed, N = c3d4_case(env, n=21)           # 10,648 nodes, ~30 k dofs
    lam, X, info = sv.lowest_modes(K, M, t, fixed, N, num_eigs=6, tol=1e-8, return_info=True, verbose=False, **KW)
    assert info["status"] == "converged"
    _, nbe = backends(env, c, t, K, M, fixed, N)
    free = nbe.mask.astype(bool)
    Kf, Mf = nbe.K[free][:, free].tocsc(), nbe.M[free][:, free].tocsc()
    ex = np.sort(sla.eigsh(Kf, 6, Mf, sigma=0, which="LM", return_eigenvectors=False))
    assert rel(lam.cpu().numpy(), ex) <= 1e-7


def test_device_driver_matches_numpy_driver_and_repeats_bitwise(env):
    el, sv, meshgen, modes, ops, MO = env
    c, t, K, M, fixed, N = c3d4_case(env, n=5)
    X0 = np.random.default_rng(11).standard_normal((3 * N, 6))
    dbe, nbe = backends(env, c, t, K, M, fixed, N)
    ld, Sd, infod = modes.lobpcg(dbe, 6, tol=1e-10, max_iter=500, X0=X0)
    ln, Sn, infon = modes.lobpcg(nbe, 6, tol=1e-10, max_iter=500, X0=X0)
    assert infod["iterations"] == infon["iterations"] and infod["status"] == "converged"
    assert np.abs(ld - ln).max() <= 1e-10 * ln.max()
    a = sv.lowest_modes(K, M, t, fixed, N, num_eigs=6, verbose=False, **KW)
    b = sv.lowest_modes(K, M, t, fixed, N, num_eigs=6, verbose=False, **KW)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    free_free = sv.lowest_modes(K, M, t, [], N, num_eigs=7, tol=1e-9, return_info=True, verbose=False, **KW)
    assert free_free[2]["status"] == "converged" and float(free_free[0][:6].abs().max()) <= 1e-8 * float(free_free[0][6])
    lam32, modes32 = sv.lowest_modes(K, M, t, fixed, N, num_eigs=2, device=DEV, dtype=torch.float32, verbose=False)
    assert lam32.dtype == torch.float32 and modes32.shape == (3 * N, 2)
    with pytest.raises(RuntimeError):
        sv.lowest_modes(K, M, t, fixed, N, device="cpu")
    with pytest.raises(ValueError):
        sv.lowest_modes(K, M, t, fixed, N, num_eigs=13, device=DEV)
