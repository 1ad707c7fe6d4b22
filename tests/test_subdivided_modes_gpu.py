"""subdivided_lowest_modes on the GPU: the two multigrid kernels of csrc/modes.cu and one device V-cycle against their numpy
restatement (tests/mg_oracle.py) on the same device-built hierarchy, and the public solver against shift-invert eigsh and against
lowest_modes (Jacobi LOBPCG) on the same finest mesh."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse.linalg as sla
import torch

from conftest import PKG

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(PKG, "solver"))

DEV = "cuda:0"
E, NU, RHO = 1.0, 0.3, 2.5


@pytest.fixture(scope="module")
def env():
    import element
    import solver
    import mg_oracle as G
    from femb200 import meshgen, multigrid
    return element, solver, G, meshgen, multigrid


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def clamp_x0(c):
    return torch.nonzero(c[:, 0].abs() < 1e-12).reshape(-1)


def free_free(c):
    return torch.zeros(0, dtype=torch.int64)


def hierarchy(env, n, levels, fixed_fn=clamp_x0, shift=0.0):
    el, sv, G, meshgen, mg = env
    c, t = meshgen.kuhn_cube(n, jitter=0.0)
    return mg.Hierarchy(c, t, levels, fixed_fn, E, NU, RHO, shift, torch.device(DEV), el)


def test_kernels_match_numpy_restatement(env):
    el, sv, G, meshgen, mg = env
    from femb200 import ops
    from femb200._lib import check, lib
    from femb200.modes import _p
    dev = torch.device(DEV)
    stream = torch.cuda.current_stream(dev).cuda_stream
    c, t = meshgen.kuhn_cube(4, jitter=0.2)
    N = c.shape[0] + 1                                        # an isolated node: an empty block row / CSR row
    plan = ops.CsrPlan(t.to(dev), N, dev)
    brow, bcol = plan.pattern(1)
    Ke = el.compute_c3d4_K_matrix(c, t, E, NU, device=dev, dtype=torch.float64)
    A = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ke, 3))
    n = 3 * N
    mask = mg.dof_mask(N, torch.nonzero(c[:, 0] == 0).reshape(-1), dev)
    dinv = A.jacobi(mask)
    An = G.MO.bsr_matrix(brow.cpu().numpy(), bcol.cpu().numpy(), A.bval.cpu().numpy()).tocsr()
    maskn, dinvn = mask.cpu().numpy(), dinv.cpu().numpy()
    rng = np.random.default_rng(3)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    for m in (1, 4, 7, 16):
        for masked in (True, False):
            mk, mkn = (mask, maskn) if masked else (None, np.ones(n, dtype=np.uint8))
            for with_x in (True, False):
                ldr, ldx, ldo = m + 3, 2 * m + 1, 3 * m
                Rh, Xh = rng.standard_normal((n, ldr)), rng.standard_normal((n, ldx))
                Rd, Xd = up(Rh), up(Xh)
                Od, Td = torch.full((n, ldo), 7.0, device=dev, dtype=torch.float64), torch.full((n, m), 7.0, device=dev, dtype=torch.float64)
                check(lib.femb_mg_smooth_bsr3(A.nb, A.nnzb, _p(A.brow), _p(A.bcol), _p(A.bval), _p(mk), _p(dinv), 0.5, m, _p(Rd, 1), ldr,
                                              _p(Xd, 2) if with_x else None, ldx, _p(Od, m), ldo, _p(Td), m, stream), "femb_mg_smooth_bsr3")
                xo, tn = G.smooth(An, mkn, dinvn, 0.5, Rh[:, 1:1 + m], Xh[:, 2:2 + m] if with_x else None)
                Oh = Od.cpu().numpy()
                assert rel(Oh[:, m:2 * m], xo) <= 1e-13 and rel(Td.cpu().numpy(), tn) <= 1e-13, (m, masked, with_x)
                assert np.all(Oh[:, :m] == 7.0) and np.all(Oh[:, 2 * m:] == 7.0)        # outside the view: untouched
                assert np.all(Oh[-3:, m:2 * m] == (Xh[-3:, 2:2 + m] if with_x else 0.0) + 0.5 * dinvn[-3:, None] * (mkn[-3:, None] * Rh[-3:, 1:1 + m]))
                # residual only, and X_out only
                T2 = torch.zeros((n, m), device=dev, dtype=torch.float64)
                check(lib.femb_mg_smooth_bsr3(A.nb, A.nnzb, _p(A.brow), _p(A.bcol), _p(A.bval), _p(mk), None, 0.5, m, _p(Rd, 1), ldr,
                                              _p(Xd, 2) if with_x else None, ldx, None, 0, _p(T2), m, stream), "femb_mg_smooth_bsr3")
                assert torch.equal(T2, Td)
    # transfers of a device hierarchy (P rows with 1-2 entries, R rows with 1 + children), plus a CSR with an empty row
    H = hierarchy(env, 3, 1)
    fine, crs = H.L[1], H.L[0]
    crow, col, val = fine.P
    crow_e = torch.cat([crow, crow[-1:]])                      # one more output node, no entries
    Pn = G.csr(tuple(a.cpu().numpy() for a in (crow_e, col, val)), (fine.nodes + 1, crs.nodes))
    Rn = G.csr(tuple(a.cpu().numpy() for a in fine.R), (crs.nodes, fine.nodes))
    for m in (1, 4, 7, 16):
        for masked in (True, False):
            for acc in (0, 1):
                Xh = rng.standard_normal((3 * crs.nodes, m + 2))
                Yh = rng.standard_normal((3 * (fine.nodes + 1), 2 * m))
                mo = torch.cat([fine.mask, torch.tensor([1, 0, 1], dtype=torch.uint8, device=dev)]) if masked else None
                Yd = up(Yh)
                check(lib.femb_mg_transfer(fine.nodes + 1, crs.nodes, col.numel(), _p(crow_e), _p(col), _p(val), _p(mo), m, _p(up(Xh), 2), m + 2,
                                           acc, _p(Yd, 1), 2 * m, stream), "femb_mg_transfer")
                mon = mo.cpu().numpy() if masked else np.ones(Yh.shape[0], dtype=np.uint8)
                ref = G.transfer(Pn, mon, Xh[:, 2:2 + m], Yh[:, 1:1 + m] if acc else None)
                got = Yd.cpu().numpy()
                assert rel(got[:, 1:1 + m], ref) <= 1e-13, (m, masked, acc)
                assert np.array_equal(got[-3:, 1:1 + m], Yh[-3:, 1:1 + m] if acc else np.zeros((3, m)))   # the empty row
                assert np.array_equal(got[:, 0], Yh[:, 0]) and np.array_equal(got[:, 1 + m:], Yh[:, 1 + m:])
                # restriction
                Fh = rng.standard_normal((3 * fine.nodes, m))
                Cd = torch.zeros((3 * crs.nodes, m), device=dev, dtype=torch.float64)
                check(lib.femb_mg_transfer(crs.nodes, fine.nodes, fine.R[1].numel(), _p(fine.R[0]), _p(fine.R[1]), _p(fine.R[2]),
                                           _p(crs.mask if masked else None), m, _p(up(Fh)), m, 0, _p(Cd), m, stream), "femb_mg_transfer")
                mcn = crs.mask.cpu().numpy() if masked else np.ones(3 * crs.nodes, dtype=np.uint8)
                assert rel(Cd.cpu().numpy(), G.transfer(Rn, mcn, Fh)) <= 1e-13


def test_device_vcycle_matches_numpy_vcycle(env):
    el, sv, G, meshgen, mg = env
    H = hierarchy(env, 3, 2)
    NH = G.NumpyHierarchy(G.from_device(H))
    f = H.L[-1].mask.cpu().numpy().astype(np.float64)[:, None]
    rng = np.random.default_rng(9)
    for k in (1, 6, 16):
        B = rng.standard_normal((f.size, k)) * f
        Vd = H.apply(torch.from_numpy(B).to(DEV)).cpu().numpy()
        assert rel(Vd, NH.apply(B)) <= 1e-12, k
        assert np.abs(Vd[f[:, 0] == 0]).max() == 0.0
    W = rng.standard_normal((f.size, 3)) * f
    V = rng.standard_normal((f.size, 3)) * f
    TV, TW = (H.apply(torch.from_numpy(X).to(DEV)).cpu().numpy() for X in (V, W))
    assert np.abs(W.T @ TV - (V.T @ TW).T).max() <= 1e-12 * np.abs(W.T @ TV).max()


def test_matches_shift_invert_eigsh(env):
    el, sv, G, meshgen, mg = env
    c, t = meshgen.kuhn_cube(4, jitter=0.0)
    lam, X, cf, tf, info = sv.subdivided_lowest_modes(c, t, 2, clamp_x0, E, NU, RHO, num_eigs=6, tol=1e-8, return_info=True,
                                                      verbose=False, device=DEV)
    assert info["status"] == "converged" and [lv["dofs"] for lv in info["levels"]] == [375, 2187, 14739] and info["shift"] == 0.0
    cfn, tfn = cf.cpu().numpy(), tf.cpu().numpy()
    N = cfn.shape[0]
    pat = G.MO.node_pattern(tfn, N)
    from oracle import fem_oracle as O
    K = G.MO.bsr_matrix(*pat, G.MO.assemble_bsr3(O.c3d4_K(cfn, tfn, E, NU), tfn, N, pat)).tocsr()
    M = G.MO.bsr_matrix(*pat, G.MO.assemble_bsr3(O.c3d4_mass(cfn, tfn, RHO), tfn, N, pat)).tocsr()
    free = G.MO.dof_mask(N, np.nonzero(np.abs(cfn[:, 0]) < 1e-12)[0]).astype(bool)
    ex = np.sort(sla.eigsh(K[free][:, free].tocsc(), 6, M[free][:, free].tocsc(), sigma=0, which="LM", return_eigenvectors=False))
    assert rel(lam.cpu().numpy(), ex) <= 1e-7
    Xh = X.cpu().numpy()
    assert np.abs(Xh[~free]).max() == 0.0 and np.abs(Xh.T @ (M @ Xh) - np.eye(6)).max() < 1e-8


def test_matches_lowest_modes_on_finest_mesh(env):
    el, sv, G, meshgen, mg = env
    c, t = meshgen.kuhn_cube(4, jitter=0.0)
    lam, X, cf, tf, info = sv.subdivided_lowest_modes(c, t, 3, clamp_x0, E, NU, RHO, return_info=True, verbose=False, device=DEV)
    assert info["status"] == "converged" and info["levels"][-1]["dofs"] == 107811
    Kl = el.compute_c3d4_K_matrix(cf, tf, E, NU, device=DEV, dtype=torch.float64)
    Ml = el.compute_c3d4_M_matrix(cf, tf, RHO, device=DEV, dtype=torch.float64)
    lj, Xj, ij = sv.lowest_modes(Kl, Ml, tf, clamp_x0(cf), cf.shape[0], num_eigs=6, return_info=True, verbose=False, device=DEV)
    assert ij["status"] == "converged"
    assert rel(lam.cpu().numpy(), lj.cpu().numpy()) <= 1e-7
    assert info["iterations"] <= 25 and 10 * info["iterations"] <= ij["iterations"], (info["iterations"], ij["iterations"])
    # same subspaces: the multigrid modes lie in the span of the Jacobi ones, per cluster of nearly equal eigenvalues
    from femb200 import ops
    plan = ops.cached_plan(tf, cf.shape[0], torch.device(DEV))
    brow, bcol = plan.pattern(1)
    Mb = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ml, 3))
    MXj = torch.stack([Mb.spmv(Xj[:, k].contiguous()) for k in range(6)], 1)
    Cm = (X.T @ MXj).cpu().numpy()                              # [6, 6] M-inner products of the two bases
    lh = lj.cpu().numpy()
    i = 0
    while i < 6:
        j = i + 1
        while j < 6 and abs(lh[j] - lh[i]) <= 1e-6 * lh[-1]:
            j += 1
        s = np.linalg.svd(Cm[i:j, i:j], compute_uv=False)
        assert s.min() >= 1 - 1e-6, (i, j, s)
        i = j


def test_repeat_is_bitwise_and_api_options(env):
    el, sv, G, meshgen, mg = env
    c, t = meshgen.kuhn_cube(3, jitter=0.1)
    a = sv.subdivided_lowest_modes(c, t, 2, clamp_x0, E, NU, RHO, verbose=False, device=DEV)
    b = sv.subdivided_lowest_modes(c, t, 2, clamp_x0, E, NU, RHO, verbose=False, device=DEV)
    # the coarse cholesky_solve runs on a fixed [n0, 16] shape every cycle; a library that changed its path between calls would show here
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    lam32, X32, _, _ = sv.subdivided_lowest_modes(c, t, 1, clamp_x0, E, NU, RHO, num_eigs=2, dtype=torch.float32, verbose=False, device=DEV)
    assert lam32.dtype == X32.dtype == torch.float32 and X32.shape[1] == 2
    lam, X, cf, tf, info = sv.subdivided_lowest_modes(c, t, 2, free_free, E, NU, RHO, num_eigs=8, tol=1e-9, shift=1.0, return_info=True,
                                                      verbose=False, device=DEV)
    assert info["status"] == "converged" and info["shift"] == 1.0
    assert float(lam[:6].abs().max()) <= 1e-8 * float(lam[6])
    lam0, _, _, _ = sv.subdivided_lowest_modes(c, t, 0, clamp_x0, E, NU, RHO, num_eigs=3, verbose=False, device=DEV)   # Cholesky only
    Kl = el.compute_c3d4_K_matrix(c, t, E, NU, device=DEV, dtype=torch.float64)
    Ml = el.compute_c3d4_M_matrix(c, t, RHO, device=DEV, dtype=torch.float64)
    lj, _ = sv.lowest_modes(Kl, Ml, t.to(DEV), clamp_x0(c), c.shape[0], num_eigs=3, verbose=False, device=DEV)
    assert rel(lam0.cpu().numpy(), lj.cpu().numpy()) <= 1e-7
    with pytest.raises(ValueError, match="shift > 0"):
        sv.subdivided_lowest_modes(c, t, 1, free_free, E, NU, RHO, verbose=False, device=DEV)
    with pytest.raises(ValueError):
        sv.subdivided_lowest_modes(c, t, 1, clamp_x0, E, NU, RHO, shift=-1.0, device=DEV)
    with pytest.raises(ValueError):
        sv.subdivided_lowest_modes(c, t, 1, clamp_x0, E, NU, RHO, num_eigs=13, device=DEV)
    with pytest.raises(ValueError, match="free dofs"):
        cb, tb = meshgen.kuhn_cube(22)                             # 34,914 free coarse dofs
        sv.subdivided_lowest_modes(cb, tb, 0, clamp_x0, E, NU, RHO, device=DEV)
    with pytest.raises(RuntimeError):
        sv.subdivided_lowest_modes(c, t, 1, clamp_x0, E, NU, RHO, device="cpu")
