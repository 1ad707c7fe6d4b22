"""Smoothed-aggregation multigrid on the GPU: the device setup (csrc/amg.cu) and femb_mg_transfer_bsr3 against the numpy restatement
(tests/amg_oracle.py), one device V-cycle against the restated cycle, amg_lowest_modes against lowest_modes and shift-invert eigsh,
and amg_buckling_modes against buckling_modes."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse.linalg as sla
import torch

import amg_oracle as A
import buckling_oracle as BO
from conftest import PKG

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(PKG, "solver"))

DEV = "cuda:0"
E, NU, RHO = 1.0, 0.3, 2.5
KW = dict(device=DEV, dtype=torch.float64)


@pytest.fixture(scope="module")
def env():
    import element
    import solver
    from femb200 import amg, meshgen, ops
    return element, solver, amg, meshgen, ops


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def h(t):
    return t.cpu().numpy()


def assembled(env, c, t, kind="c3d4", fixed_x0=True):
    el, sv, amg, meshgen, ops = env
    K_loc = {"c3d4": el.compute_c3d4_K_matrix, "c3d10": el.compute_c3d10_K_matrix, "c3d8": el.compute_c3d8_K_matrix}[kind](c, t, E, NU, **KW)
    M_loc = {"c3d4": el.compute_c3d4_M_matrix, "c3d10": el.compute_c3d10_M_matrix, "c3d8": el.compute_c3d8_M_matrix}[kind](c, t, RHO, **KW)
    N = c.shape[0]
    plan = ops.CsrPlan(t, N, DEV)
    brow, bcol = plan.pattern(1)
    K = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(K_loc, 3))
    M = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(M_loc, 3))
    fixed = torch.nonzero(c[:, 0] == 0).reshape(-1) if fixed_x0 else torch.zeros(0, dtype=torch.long)
    return K_loc, M_loc, K, M, fixed


def test_setup_matches_restatement_and_repeats_bitwise(env):
    el, sv, amg, meshgen, ops = env
    c, t = meshgen.kuhn_cube(12, jitter=0.2)
    _, _, K, M, fixed = assembled(env, c, t)
    from femb200 import multigrid
    mask = multigrid.dof_mask(c.shape[0], fixed, DEV)
    H = amg.AmgHierarchy(K, mask, c, K=K, M=M, coarse_dofs=150)
    H2 = amg.AmgHierarchy(K, mask, c, K=K, M=M, coarse_dofs=150)
    NH = A.NumpyAmg((h(K.brow), h(K.bcol), h(K.bval)), h(mask), c.numpy(), coarse_dofs=150)
    assert len(H.L) == len(NH.levels) >= 3
    for k, nl in enumerate(NH.levels):
        dl, dl2 = H.L[-1 - k], H2.L[-1 - k]
        assert np.array_equal(h(dl.mask), nl["mask"])
        for name, T in (("A", dl.A), ("P", dl.P), ("R", dl.R)):
            ref = nl["T"] if name == "A" else nl.get(name)
            if ref is None:
                assert T is None
                continue
            assert np.array_equal(h(T.brow), ref[0]) and np.array_equal(h(T.bcol), ref[1]), (k, name)
            assert rel(h(T.bval), ref[2]) <= 1e-13, (k, name, rel(h(T.bval), ref[2]))
            T2 = getattr(dl2, name)
            assert torch.equal(T.bval, T2.bval) and torch.equal(T.bcol, T2.bcol), (k, name)
    # aggregates and the tentative prolongator of the finest level
    agg, n_agg = amg.aggregate(K, mask)
    agg_n, n_n = A.aggregate(h(K.brow), h(K.bcol), h(mask))
    assert n_agg == n_n and np.array_equal(h(agg), agg_n)
    Pt, Bc, mc, cc = amg.tentative(agg, n_agg, mask, c.to(DEV))
    (pr, pc, pv), Bcn, mcn, ccn = A.tentative(agg_n, n_n, h(mask), c.numpy())
    assert np.array_equal(h(Pt.brow), pr) and np.array_equal(h(Pt.bcol), pc) and np.array_equal(h(mc), mcn)
    assert rel(h(Pt.bval), pv) <= 1e-13 and rel(h(Bc), Bcn) <= 1e-13 and rel(h(cc), ccn) <= 1e-15
    # a coarse level: the carried modes re-centred on the coarse aggregates
    crs = H.L[-2]
    agg2, n2 = amg.aggregate(crs.A, crs.mask)
    Pt2, Bc2, mc2, _ = amg.tentative(agg2, n2, crs.mask, cc, Bc)
    (pr2, pc2, pv2), Bcn2, mcn2, _ = A.tentative(h(agg2), n2, h(crs.mask), ccn, Bcn)
    assert np.array_equal(h(Pt2.bcol), pc2) and np.array_equal(h(mc2), mcn2)
    assert rel(h(Pt2.bval), pv2) <= 1e-12 and rel(h(Bc2), Bcn2) <= 1e-12


def test_transfer_and_vcycle_match_restatement(env):
    el, sv, amg, meshgen, ops = env
    from femb200 import multigrid
    c, t = meshgen.kuhn_cube(10, jitter=0.2)
    _, _, K, M, fixed = assembled(env, c, t)
    mask = multigrid.dof_mask(c.shape[0], fixed, DEV)
    H = amg.AmgHierarchy(K, mask, c, K=K, M=M, coarse_dofs=150)
    NH = A.NumpyAmg((h(K.brow), h(K.bcol), h(K.bval)), h(mask), c.numpy(), coarse_dofs=150)
    fine, crs = H.L[-1], H.L[-2]
    rng = np.random.default_rng(3)
    for m in (1, 5, 16):
        X = rng.standard_normal((fine.n, m))
        fine.t[:, :m].copy_(torch.from_numpy(X))
        fine.restrict(crs, m, fine.t, H.stream)
        assert rel(h(crs.b[:, :m]), A.transfer(NH.levels[0]["R"], NH.levels[1]["mask"], X, fine.nodes)) <= 1e-13
        Xc = rng.standard_normal((crs.n, m))
        Y = rng.standard_normal((fine.n, m))
        crs.x[:, :m].copy_(torch.from_numpy(Xc))
        fine.y[:, :m].copy_(torch.from_numpy(Y))
        fine.prolong(crs, m, crs.x, fine.y, H.stream)
        assert rel(h(fine.y[:, :m]), A.transfer(NH.levels[0]["P"], fine.mask.cpu().numpy(), Xc, crs.nodes, Y)) <= 1e-13
    f = h(mask).astype(np.float64)[:, None]
    B = rng.standard_normal((fine.n, 6)) * f
    Vd = h(H.apply(torch.from_numpy(B).to(DEV)))
    assert rel(Vd, NH.apply(B)) <= 1e-11
    assert np.array_equal(Vd, h(H.apply(torch.from_numpy(B).to(DEV))))


def check_against_lowest_modes(env, c, t, kind, num_eigs=6):
    el, sv, amg, meshgen, ops = env
    K_loc, M_loc, K, M, fixed = assembled(env, c, t, kind)
    N = c.shape[0]
    lam, X, info = sv.amg_lowest_modes(c, K_loc, M_loc, t.to(DEV), fixed, num_eigs=num_eigs, tol=1e-10, max_iter=300, return_info=True,
                                       verbose=False, **KW)
    assert info["status"] == "converged", info["iterations"]
    lj, Xj = sv.lowest_modes(K_loc, M_loc, t.to(DEV), fixed, N, num_eigs=num_eigs, tol=1e-10, max_iter=20000, verbose=False, **KW)
    assert rel(h(lam), h(lj)) <= 1e-7
    from oracle import modes_oracle as MO
    mask = MO.dof_mask(N, h(fixed))
    free = mask.astype(bool)
    Kf = MO.bsr_matrix(h(K.brow), h(K.bcol), h(K.bval)).tocsr()[free][:, free].tocsc()
    Mf = MO.bsr_matrix(h(M.brow), h(M.bcol), h(M.bval)).tocsr()
    ex = np.sort(sla.eigsh(Kf, num_eigs, Mf[free][:, free].tocsc(), sigma=0, which="LM", return_eigenvectors=False))
    assert rel(h(lam), ex) <= 1e-7
    Xh = h(X)
    assert np.abs(Xh[~free]).max() == 0.0
    assert np.abs(Xh.T @ (Mf @ Xh) - np.eye(num_eigs)).max() <= 1e-9
    return lam, X, info


def test_amg_lowest_modes_c3d4_c3d10_c3d8(env):
    el, sv, amg, meshgen, ops = env
    c, t = meshgen.kuhn_cube(16, jitter=0.2)
    lam, X, info = check_against_lowest_modes(env, c, t, "c3d4")
    assert len(info["levels"]) >= 2 and info["setup_ms"]["spgemm"] > 0
    lam2, X2 = sv.amg_lowest_modes(c, el.compute_c3d4_K_matrix(c, t, E, NU, **KW), el.compute_c3d4_M_matrix(c, t, RHO, **KW), t.to(DEV),
                                   torch.nonzero(c[:, 0] == 0).reshape(-1), num_eigs=6, tol=1e-10, max_iter=300, verbose=False, **KW)
    assert torch.equal(lam, lam2) and torch.equal(X, X2)
    c, t = meshgen.tet10_cube(10, jitter=0.1)
    check_against_lowest_modes(env, c, t, "c3d10")
    c, hx = meshgen.hex_cube(18, jitter=0.1)
    check_against_lowest_modes(env, c, hx, "c3d8", num_eigs=5)


def test_free_free_needs_a_shift(env):
    el, sv, amg, meshgen, ops = env
    c, t = meshgen.kuhn_cube(16, jitter=0.2)
    K_loc, M_loc, K, M, _ = assembled(env, c, t, fixed_x0=False)
    none = torch.zeros(0, dtype=torch.long)
    lam, X, info = sv.amg_lowest_modes(c, K_loc, M_loc, t.to(DEV), none, num_eigs=8, tol=1e-9, shift=1.0, return_info=True, verbose=False, **KW)
    assert info["status"] == "converged"
    lam = h(lam)
    assert np.abs(lam[:6]).max() <= 1e-8 * lam[6]
    with pytest.raises(ValueError, match="shift > 0"):
        sv.amg_lowest_modes(c, K_loc, M_loc, t.to(DEV), none, num_eigs=6, verbose=False, **KW)


@pytest.mark.parametrize("quadratic", [False, True], ids=["c3d4", "c3d10"])
def test_amg_buckling_matches_buckling_modes(env, quadratic):
    el, sv, amg, meshgen, ops = env
    c, t = BO.column(2, quadratic=quadratic)
    F = BO.top_load(c)
    fixed = BO.clamp_base(c)
    lam, X, u, info = sv.amg_buckling_modes(c, t, F, fixed, E, NU, num_eigs=4, tol=1e-10, return_info=True, verbose=False, **KW)
    assert info["status"] == "converged"
    lj, Xj, uj = sv.buckling_modes(c, t, F, fixed, E, NU, num_eigs=4, tol=1e-10, max_iter=40000, static_max_iter=200000, verbose=False, **KW)
    assert rel(h(lam), h(lj)) <= 1e-6
    assert rel(h(u), h(uj)) <= 1e-7
    lam2, X2, u2 = sv.amg_buckling_modes(c, t, F, fixed, E, NU, num_eigs=4, tol=1e-10, verbose=False, **KW)
    assert torch.equal(lam, lam2) and torch.equal(X, X2)
    if not quadratic:   # the refinement V-cycle on a refined column against AMG on the same mesh, passed flat
        ls, _, _, cf, tf = sv.subdivided_buckling_modes(*BO.column(1), 1, lambda cc, tt: BO.top_load(cc.cpu().numpy()),
                                                        lambda cc: BO.clamp_base(cc.cpu().numpy()), E, NU, num_eigs=4, tol=1e-10,
                                                        verbose=False, **KW)
        la = sv.amg_buckling_modes(cf, tf, BO.top_load(h(cf)), BO.clamp_base(h(cf)), E, NU, num_eigs=4, tol=1e-10, verbose=False, **KW)[0]
        assert rel(h(la), h(ls)) <= 1e-6
    with pytest.raises(ValueError, match="free-free"):
        sv.amg_buckling_modes(c, t, F, [], E, NU, verbose=False, **KW)
    with pytest.raises(ValueError, match="zero"):
        sv.amg_buckling_modes(c, t, np.zeros_like(F), fixed, E, NU, verbose=False, **KW)
