"""lowest_modes without a GPU: the LOBPCG driver (femb200/modes.py) on the numpy restatement of its four block kernels
(oracle/modes_oracle.py) against dense generalized eigensolves, and argument validation of the new C ABI entries."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sl

from femb200 import meshgen, modes
from oracle import fem_oracle as O
from oracle import modes_oracle as MO


def cantilever(n=4, fixed_face=True, rho=2.5):
    c, t = meshgen.kuhn_cube(n, jitter=0.2)
    c, t = c.numpy(), t.numpy()
    N = c.shape[0]
    pat = MO.node_pattern(t, N)
    kv = MO.assemble_bsr3(O.c3d4_K(c, t, 1.0, 0.3), t, N, pat)
    mv = MO.assemble_bsr3(O.c3d4_mass(c, t, rho), t, N, pat)
    fixed = np.nonzero(c[:, 0] == 0)[0] if fixed_face else np.array([], dtype=np.int64)
    return c, MO.NumpyBackend(*pat, kv, mv, MO.dof_mask(N, fixed))


def dense_pencil(be):
    free = be.mask.astype(bool)
    return free, be.K.toarray()[np.ix_(free, free)], be.M.toarray()[np.ix_(free, free)]


def assert_same_modes(lam, X, ex, V, Md, tol_lam, tol_sub):
    """Eigenvalues within tol_lam relative to the spectrum's scale; subspaces compared per cluster (eigenvalues closer than 1e-6
    relative) by principal angles, so degenerate modes and signs do not matter."""
    k = lam.size
    scale = max(abs(ex[k - 1]), abs(ex[k]))
    assert np.abs(lam - ex[:k]).max() <= tol_lam * scale, (lam, ex[:k])
    i = 0
    while i < k:
        j = i + 1
        while j < len(ex) and abs(ex[j] - ex[i]) <= 1e-6 * scale:
            j += 1
        Vc, Xc = V[:, i:min(j, len(ex))], X[:, i:min(j, k)]
        # M-orthonormal bases: sin of the largest principal angle = |(I - Vc Vc^T M) Xc|_M
        R = Xc - Vc @ (Vc.T @ (Md @ Xc))
        assert np.sqrt(max(np.linalg.eigvalsh(R.T @ Md @ R).max(), 0.0)) <= tol_sub, (i, j)
        i = j


def test_cantilever_matches_dense_eigh():
    _, be = cantilever()
    lam, S, info = modes.lobpcg(be, 6, tol=1e-10, max_iter=500)
    assert info["status"] == "converged" and info["residuals"].max() <= 1e-10
    free, Kd, Md = dense_pencil(be)
    ex, V = sl.eigh(Kd, Md)
    X = S[:, :6]
    assert np.abs(X[~free]).max() == 0.0
    assert np.abs(X.T @ (be.M @ X) - np.eye(6)).max() < 1e-10
    assert_same_modes(lam, X[free], ex, V, Md, 1e-8, 1e-6)
    assert np.allclose(info["freq_hz"], np.sqrt(lam) / (2 * np.pi))


def test_free_free_rigid_body_modes():
    c, be = cantilever(fixed_face=False)
    lam, S, info = modes.lobpcg(be, 7, tol=1e-10, max_iter=500)
    assert info["status"] == "converged"
    assert np.abs(lam[:6]).max() <= 1e-8 * lam[6]
    X = S[:, :6]
    rb = np.zeros((c.shape[0], 3, 6))
    for d in range(3):
        rb[:, d, d] = 1.0                                        # translations
    for k, (a, b) in enumerate(((1, 2), (2, 0), (0, 1))):       # rotations
        rb[:, a, 3 + k] = -c[:, b]
        rb[:, b, 3 + k] = c[:, a]
    rb = rb.reshape(-1, 6)
    # M-projection residual of the rigid-body vectors onto the mode span, relative to their M-norm
    P = rb - X @ (X.T @ (be.M @ rb))
    ratio = np.sqrt(np.diag(P.T @ (be.M @ P)) / np.diag(rb.T @ (be.M @ rb)))
    assert ratio.max() <= 1e-6, ratio


def test_nearly_dependent_start_block_and_restart():
    """A start block whose columns are nearly (or exactly) the same vector still converges to the dense result; and the
    Rayleigh-Ritz step drops P (one restart) when the P block is numerically dependent on [X W]."""
    _, be = cantilever()
    free, Kd, Md = dense_pencil(be)
    ex, V = sl.eigh(Kd, Md)
    rng = np.random.default_rng(3)
    X0 = np.zeros((be.n, 6))
    X0[free] = V[:, [0]] + 1e-9 * rng.standard_normal((free.sum(), 6))
    X0[:, 5] = X0[:, 4]
    lam, S, info = modes.lobpcg(be, 6, tol=1e-10, max_iter=500, X0=X0)
    assert info["status"] == "converged"
    assert_same_modes(lam, S[free, :6], ex, V, Md, 1e-8, 1e-6)

    # basis [X W P] with P = W C + 1e-12 noise: the M-Gram of the whole basis is numerically singular
    m = 4
    B = rng.standard_normal((60, 3 * m))
    B[:, 2 * m:] = B[:, m:2 * m] @ rng.standard_normal((m, m)) + 1e-12 * rng.standard_normal((60, m))
    A = np.diag(np.arange(1.0, 61.0))
    GK, GM = B.T @ A @ B, B.T @ B
    lam3, CX, CP, dropped = modes._rayleigh_ritz(GK, GM, [(np.arange(m), "x"), (m + np.arange(m), "w"), (2 * m + np.arange(m), "p")], m)
    lam2, _, _, dropped2 = modes._rayleigh_ritz(GK[:2 * m, :2 * m], GM[:2 * m, :2 * m], [(np.arange(m), "x"), (m + np.arange(m), "w")], m)
    assert dropped and not dropped2
    assert np.abs(lam3 - lam2).max() <= 1e-12 * lam2.max()
    assert np.abs(CX[2 * m:]).max() == 0.0 and np.abs((B @ CX).T @ (B @ CX) - np.eye(m)).max() < 1e-10


def test_max_iter_returns_current_ritz_pairs():
    _, be = cantilever()
    lam, S, info = modes.lobpcg(be, 3, tol=1e-14, max_iter=5)
    assert info["status"] == "maxiter" and info["iterations"] == 5 and lam.shape == (3,) and np.all(np.diff(lam) >= 0)
    assert modes.block_width(1) == 4 and modes.block_width(6) == 8 and modes.block_width(12) == 16


def test_new_entry_points_validate_arguments_without_gpu():
    from femb200 import _lib
    L = _lib.lib
    buf = (ctypes.c_double * 4096)()
    p = ctypes.addressof(buf)
    q = p + 8 * 2048
    lam = (ctypes.c_double * 16)()
    C = (ctypes.c_double * (48 * 16))()

    def err(rc, word):
        assert rc == 1 and word in L.femb_last_error(), L.femb_last_error()

    # femb_spmm_bsr3: m range, null pointers, ld < m, overlapping output
    err(L.femb_spmm_bsr3(1, 1, p, p, p, None, None, 17, p, 17, q, None, 17, None), b"m <= 16")
    err(L.femb_spmm_bsr3(1, 1, p, p, p, None, None, 0, p, 4, q, None, 4, None), b"m <= 16")
    err(L.femb_spmm_bsr3(1, 1, None, p, p, None, None, 4, p, 4, q, None, 4, None), b"non-null")
    err(L.femb_spmm_bsr3(1, 1, p, p, p, p, None, 4, p, 4, q, None, 4, None), b"mval and YM")
    err(L.femb_spmm_bsr3(1, 1, p, p, p, None, None, 4, p, 3, q, None, 4, None), b"ldx")
    err(L.femb_spmm_bsr3(1, 1, p, p, p, None, None, 4, p, 8, p + 8 * 8, None, 8, None), b"overlap")
    # femb_mb_gram: ka / kb range, null pointers, ld < k, G overlapping an input
    err(L.femb_mb_gram(10, 49, p, 49, 4, p, 4, q, None), b"ka, kb <= 48")
    err(L.femb_mb_gram(10, 4, p, 4, 49, p, 49, q, None), b"ka, kb <= 48")
    err(L.femb_mb_gram(10, 4, None, 4, 4, p, 4, q, None), b"non-null")
    err(L.femb_mb_gram(10, 4, p, 3, 4, p, 4, q, None), b"lda")
    err(L.femb_mb_gram(10, 4, p, 4, 4, p, 4, p + 8, None), b"overlap")
    # femb_mb_combine: k / mc range, null pointers, ld < k, overlapping output (interleaved views of one buffer are allowed)
    err(L.femb_mb_combine(10, 49, p, 49, 4, C, 0.0, q, 4, None), b"k <= 48")
    err(L.femb_mb_combine(10, 8, p, 8, 17, C, 0.0, q, 17, None), b"mc <= 16")
    err(L.femb_mb_combine(10, 8, p, 8, 4, None, 0.0, q, 4, None), b"non-null")
    err(L.femb_mb_combine(10, 8, p, 7, 4, C, 0.0, q, 4, None), b"ldx")
    err(L.femb_mb_combine(10, 8, p, 12, 4, C, 0.0, p + 8 * 7, 12, None), b"overlap")
    # femb_lobpcg_residual: m / na range, null pointers, ld < m, W overlapping X
    err(L.femb_lobpcg_residual(10, 17, p, 17, q, q, 17, lam, p, 0, None, None, 1, p, None), b"m <= 16")
    err(L.femb_lobpcg_residual(10, 4, p, 4, q, q, 4, lam, p, 5, p, q, 4, p, None), b"na <= m")
    err(L.femb_lobpcg_residual(10, 4, p, 4, q, q, 4, None, p, 0, None, None, 1, p, None), b"non-null")
    err(L.femb_lobpcg_residual(10, 4, p, 3, q, q, 4, lam, p, 0, None, None, 1, p, None), b"ldx")
    err(L.femb_lobpcg_residual(10, 4, p, 12, q, q, 12, lam, q, 4, p, p + 8 * 2, 12, q, None), b"W overlaps")
