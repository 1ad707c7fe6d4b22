"""subdivided_lowest_modes without a GPU: the LOBPCG driver (femb200/modes.py) with the numpy restatement of the multigrid V-cycle
(tests/mg_oracle.py) against dense eigensolves and the Jacobi backend, properties of the cycle, and argument validation of the
two multigrid C ABI entries."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sl

import mg_oracle as G
from femb200 import meshgen, modes
from oracle import modes_oracle as MO
from test_lowest_modes_cpu import assert_same_modes

E, NU, RHO = 1.0, 0.3, 2.5


def clamp_x0(c):
    return np.nonzero(np.abs(c[:, 0]) < 1e-12)[0]


def free_free(c):
    return np.array([], dtype=np.int64)


def coarse(n):
    c, t = meshgen.kuhn_cube(n, jitter=0.0)
    return c.numpy(), t.numpy()


@pytest.fixture(scope="module")
def cube4():
    """kuhn_cube(4) refined 1, 2 and 3 times (2,187 / 14,739 / 107,811 dofs), x = 0 face clamped."""
    c, t = coarse(4)
    return {L: G.numpy_hierarchy(c, t, L, clamp_x0, E, NU, RHO) for L in (1, 2, 3)}


def jacobi_backend(levels, kval, mval):
    top = levels[-1]
    return MO.NumpyBackend(top["brow"], top["bcol"], kval, mval, top["mask"])


def test_multigrid_driver_matches_dense_eigh():
    c, t = coarse(3)
    levels, kval, mval, cf, tf = G.numpy_hierarchy(c, t, 2, clamp_x0, E, NU, RHO)
    be = G.NumpyMultilevelBackend(levels, kval, mval)
    assert be.n == 6591
    lam, S, info = modes.lobpcg(be, 6, tol=1e-10, max_iter=200)
    assert info["status"] == "converged"
    free = be.mask.astype(bool)
    Kd, Md = be.K.toarray()[np.ix_(free, free)], be.M.toarray()[np.ix_(free, free)]
    ex, V = sl.eigh(Kd, Md, subset_by_index=[0, 11])
    X = S[:, :6]
    assert np.abs(X[~free]).max() == 0.0
    assert np.abs(X.T @ (be.M @ X) - np.eye(6)).max() < 1e-10
    assert_same_modes(lam, X[free], ex, V, Md, 1e-8, 1e-6)


def test_iterations_do_not_grow_with_refinement(cube4):
    its = []
    for L in (1, 2, 3):
        levels, kval, mval, cf, tf = cube4[L]
        lam, S, info = modes.lobpcg(G.NumpyMultilevelBackend(levels, kval, mval), 6, tol=1e-8, max_iter=200)
        assert info["status"] == "converged", L
        its.append(info["iterations"])
    assert max(its) <= 25 and max(its) - min(its) <= 4, its


def test_far_fewer_iterations_than_jacobi(cube4):
    levels, kval, mval, cf, tf = cube4[2]
    lm, _, im = modes.lobpcg(G.NumpyMultilevelBackend(levels, kval, mval), 6, tol=1e-8, max_iter=200)
    lj, _, ij = modes.lobpcg(jacobi_backend(levels, kval, mval), 6, tol=1e-8, max_iter=2000)
    assert im["status"] == ij["status"] == "converged"
    assert 5 * im["iterations"] <= ij["iterations"], (im["iterations"], ij["iterations"])
    assert np.abs(lm - lj).max() <= 1e-7 * lj.max()


def test_vcycle_is_symmetric(cube4):
    levels, kval, mval, cf, tf = cube4[2]
    H = G.NumpyHierarchy(levels)
    f = levels[-1]["mask"].astype(np.float64)[:, None]
    rng = np.random.default_rng(4)
    V, W = rng.standard_normal((f.size, 3)) * f, rng.standard_normal((f.size, 3)) * f
    TV, TW = H.apply(V), H.apply(W)
    a, b = W.T @ TV, V.T @ TW
    assert np.abs(a - b.T).max() <= 1e-12 * np.abs(a).max()
    assert np.all(np.einsum("ij,ij->j", V, TV) > 0)                # and positive definite on these vectors
    assert np.abs(TV[f[:, 0] == 0]).max() == 0.0


def test_levels_zero_is_the_coarse_solve():
    c, t = coarse(3)
    levels, kval, mval, cf, tf = G.numpy_hierarchy(c, t, 0, clamp_x0, E, NU, RHO)
    be = G.NumpyMultilevelBackend(levels, kval, mval)
    lam, S, info = modes.lobpcg(be, 4, tol=1e-10, max_iter=50)
    assert info["status"] == "converged" and info["iterations"] <= 12     # K^-1 as the preconditioner
    free = be.mask.astype(bool)
    ex = sl.eigh(be.K.toarray()[np.ix_(free, free)], be.M.toarray()[np.ix_(free, free)], eigvals_only=True)
    assert np.abs(lam - ex[:4]).max() <= 1e-8 * ex[4]


def test_free_free_with_shift_gives_rigid_body_modes():
    c, t = coarse(4)
    levels, kval, mval, cf, tf = G.numpy_hierarchy(c, t, 1, free_free, E, NU, RHO, shift=1.0)
    be = G.NumpyMultilevelBackend(levels, kval, mval)
    lam, S, info = modes.lobpcg(be, 8, tol=1e-9, max_iter=200)
    assert info["status"] == "converged"
    assert np.abs(lam[:6]).max() <= 1e-8 * lam[6]
    X = S[:, :6]
    rb = np.zeros((cf.shape[0], 3, 6))
    for d in range(3):
        rb[:, d, d] = 1.0
    for k, (a, b) in enumerate(((1, 2), (2, 0), (0, 1))):
        rb[:, a, 3 + k] = -cf[:, b]
        rb[:, b, 3 + k] = cf[:, a]
    rb = rb.reshape(-1, 6)
    P = rb - X @ (X.T @ (be.M @ rb))
    ratio = np.sqrt(np.diag(P.T @ (be.M @ P)) / np.diag(rb.T @ (be.M @ rb)))
    assert ratio.max() <= 1e-6, ratio


def test_free_free_without_shift_is_refused():
    c, t = coarse(3)
    levels, kval, mval, cf, tf = G.numpy_hierarchy(c, t, 1, free_free, E, NU, RHO, shift=0.0)
    with pytest.raises(ValueError, match="shift > 0"):
        G.NumpyMultilevelBackend(levels, kval, mval)


def test_refinement_and_transfers():
    """numpy refine_once: 8 children per tet, total volume kept, P reproduces linear fields, R = P^T."""
    c, t = coarse(2)
    c2, t2, par = G.refine_once(c, t)
    assert t2.shape == (8 * t.shape[0], 4) and c2.shape[0] == c.shape[0] + par.shape[0]
    from oracle import fem_oracle as O
    assert abs(np.abs(O.tet_volumes(c2, t2)).sum() - np.abs(O.tet_volumes(c, t)).sum()) < 1e-12
    (pc, pcol, pv), (rc, rcol, rv) = G.prolongation(par, c.shape[0])
    P = G.csr((pc, pcol, pv), (c2.shape[0], c.shape[0]))
    R = G.csr((rc, rcol, rv), (c.shape[0], c2.shape[0]))
    assert np.abs(P @ c - c2).max() < 1e-14 and (abs(P.T - R) > 0).nnz == 0
    mask = np.ones(3 * c2.shape[0], dtype=np.uint8)
    X = np.random.default_rng(1).standard_normal((3 * c.shape[0], 5))
    assert np.abs(G.transfer(P, mask, X) - np.kron(P.toarray(), np.eye(3)) @ X).max() < 1e-14


def test_multigrid_entry_points_validate_arguments_without_gpu():
    from femb200 import _lib
    L = _lib.lib
    buf = (ctypes.c_double * 8192)()
    p = ctypes.addressof(buf)
    q, r = p + 8 * 2048, p + 8 * 4096

    def err(rc, word):
        assert rc == 1 and word in L.femb_last_error(), L.femb_last_error()

    # femb_mg_smooth_bsr3(nb, nnzb, brow, bcol, aval, mask, dinv, omega, m, R, ldr, X_in, ldx, X_out, ldo, Res, ldres, stream)
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 17, p, 17, q, 17, r, 17, None, 0, None), b"m <= 16")
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 0, p, 4, q, 4, r, 4, None, 0, None), b"m <= 16")
    err(L.femb_mg_smooth_bsr3(2, 1, None, p, p, None, p, 0.5, 4, p, 4, q, 4, r, 4, None, 0, None), b"non-null")
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 4, p, 4, q, 4, None, 0, None, 0, None), b"non-null")   # no output
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, None, 0.5, 4, p, 4, q, 4, r, 4, None, 0, None), b"dinv")      # X_out without dinv
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 4, p, 3, q, 4, r, 4, None, 0, None), b"ldr")
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 4, p, 4, q, 4, r, 4, r + 8 * 2, 8, None), b"overlap")
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 4, p, 4, q, 8, q + 8 * 2, 8, None, 0, None), b"overlap")  # X_out meets X_in
    err(L.femb_mg_smooth_bsr3(2, 1, p, p, p, None, p, 0.5, 4, q, 4, None, 0, q, 4, None, 0, None), b"overlap")       # X_out = R
    assert L.femb_mg_smooth_bsr3(0, 0, p, p, p, None, p, 0.5, 4, p, 4, None, 0, q, 4, None, 0, None) == 0           # empty: no launch
    # femb_mg_transfer(n_out, n_in, nnz, crow, col, val, mask_out, m, X, ldx, accumulate, Y, ldy, stream)
    err(L.femb_mg_transfer(2, 2, 2, p, p, p, None, 17, q, 17, 0, r, 17, None), b"m <= 16")
    err(L.femb_mg_transfer(2, 2, 2, None, p, p, None, 4, q, 4, 0, r, 4, None), b"non-null")
    err(L.femb_mg_transfer(2, 2, 2, p, p, p, None, 4, q, 4, 0, None, 4, None), b"non-null")
    err(L.femb_mg_transfer(2, 2, 2, p, p, p, None, 4, q, 3, 0, r, 4, None), b"ldx")
    err(L.femb_mg_transfer(2, 2, 2, p, p, p, None, 4, q, 4, 2, r, 4, None), b"accumulate")
    err(L.femb_mg_transfer(2, 2, 2, p, p, p, None, 4, q, 4, 0, q + 8 * 8, 4, None), b"overlaps")
    assert L.femb_mg_transfer(0, 2, 0, p, p, p, None, 4, q, 4, 0, r, 4, None) == 0
