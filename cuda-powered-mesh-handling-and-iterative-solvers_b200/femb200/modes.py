"""LOBPCG for the lowest eigenpairs of K x = lam M x (3 dofs per node, K and M on one 3x3 block pattern).

Knyazev's locally optimal block preconditioned CG with a Jacobi preconditioner and the robustness steps of Hetmaniuk & Lehoucq
(2006) and Duersch et al. (2018): the basis S = [X | W | P] is M-orthonormalised block by block (Cholesky-QR done twice), converged
columns are soft-locked (their residuals leave W) and P is dropped for one iteration (a restart) when its block is numerically
dependent on [X W].  The block carries m = roundup(num_eigs + 2, 4) <= 16 columns; the guard columns speed up the last wanted pair.

Every n-long operation goes through a backend with four methods -- `spmm`, `gram`, `combine`, `residual` -- plus `zeros`,
`upload` and `host` for memory.  `DeviceBackend` calls the block kernels of csrc/modes.cu; the numpy restatement used by the tests
is oracle/modes_oracle.py.  Per iteration the host receives one copy (both 3m x 3m Grams and the residual norms) and solves the
Rayleigh-Ritz problem; the Ritz coefficients go back as kernel arguments.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch

from ._lib import check, lib

START_SEED = 20241020        # default start block: fixed seed, so repeated calls are bit-identical
DEPENDENT_PIVOT = 1e-7       # a block whose projected, column-normalised Gram has a Cholesky pivot below this is dependent


def block_width(num_eigs):
    return min(16, -(-(num_eigs + 2) // 4) * 4)


def start_block(n, m, X0=None):
    """[n, m] host start block: the columns of X0 (optional), the rest from the fixed-seed generator."""
    X = np.random.default_rng(START_SEED).standard_normal((n, m))
    if X0 is not None:
        X0 = np.asarray(X0, dtype=np.float64).reshape(n, -1)
        X[:, :X0.shape[1]] = X0
    return X


# ----------------------------------------------------------------------------------------------------------- device backend

def _p(t, c0=0):
    return C.c_void_p(t.data_ptr() + 8 * c0) if t is not None else C.c_void_p(0)


class DeviceBackend:
    """The block kernels of csrc/modes.cu on [n, ld] row-major fp64 CUDA tensors.  K, M: ops.Bsr3 on one pattern; mask: uint8 per
    dof (0 = fixed)."""

    def __init__(self, K, M, mask):
        assert K.brow is M.brow or torch.equal(K.bcol, M.bcol), "K and M must share one block pattern"
        self.K, self.M, self.mask, self.dev = K, M, mask, K.dev
        self.n = 3 * K.nb
        self.stream = torch.cuda.current_stream(self.dev).cuda_stream
        self.dinv = K.jacobi(mask)
        ones = torch.ones(self.n, device=self.dev, dtype=torch.float64)
        # |A|_1 = |A|_inf (symmetric) = max of |A| 1, with the library's own SpMV (deterministic)
        self.norm_K, self.norm_M = (float(type(A)(A.brow, A.bcol, A.bval.abs()).spmv(ones).max()) for A in (K, M))

    def zeros(self, rows, cols):
        return torch.zeros((rows, cols), device=self.dev, dtype=torch.float64)

    def upload(self, a):
        return torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)

    def host(self, t):
        return t.cpu().numpy()

    def mask_host(self):
        return self.mask.cpu().numpy()

    def spmm(self, X, c0, k, YK, YM):
        """YK[:, c0:c0+k] = K X[:, c0:c0+k], YM likewise with M (one pass); rows of fixed dofs are zero."""
        K, M = self.K, self.M
        with torch.cuda.device(self.dev):
            check(lib.femb_spmm_bsr3(K.nb, K.nnzb, _p(K.brow), _p(K.bcol), _p(K.bval), _p(M.bval), _p(self.mask), k, _p(X, c0), X.shape[1],
                                     _p(YK, c0), _p(YM, c0), YK.shape[1], self.stream), "femb_spmm_bsr3")

    def gram(self, A, B, k, G):
        """G[:k*k] = A[:, :k]^T B[:, :k] (device)."""
        with torch.cuda.device(self.dev):
            check(lib.femb_mb_gram(A.shape[0], k, _p(A), A.shape[1], k, _p(B), B.shape[1], _p(G), self.stream), "femb_mb_gram")

    def combine(self, X, k, Cm, Y, c0, beta=0.0):
        """Y[:, c0:c0+mc] = beta Y[:, c0:c0+mc] + X[:, :k] Cm (Cm [k, mc] host)."""
        Cm = np.ascontiguousarray(Cm, dtype=np.float64)
        with torch.cuda.device(self.dev):
            check(lib.femb_mb_combine(X.shape[0], k, _p(X), X.shape[1], Cm.shape[1], Cm.ctypes.data_as(C.POINTER(C.c_double)), float(beta),
                                      _p(Y, c0), Y.shape[1], self.stream), "femb_mb_combine")

    def residual(self, X, KX, MX, m, lam, active, na, W, c0, norms):
        """R = KX - MX diag(lam) over the first m columns; norms[:m] = |r_j|^2, norms[m:2m] = |x_j|^2; W[:, c0+a] = D^-1 r_active[a]."""
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        with torch.cuda.device(self.dev):
            check(lib.femb_lobpcg_residual(X.shape[0], m, _p(X), X.shape[1], _p(KX), _p(MX), KX.shape[1], lam.ctypes.data_as(C.POINTER(C.c_double)),
                                           _p(self.dinv), na, _p(active), _p(W, c0), W.shape[1], _p(norms), self.stream),
                  "femb_lobpcg_residual")

    def active_list(self, cols):
        return torch.tensor(cols, device=self.dev, dtype=torch.int32)


# ------------------------------------------------------------------------------------------------------ small-space algebra

def _orthonormalise(GM, V, Q, allow_drop, pivot=DEPENDENT_PIVOT):
    """M-orthonormalise the basis directions V (coefficients over S) against Q (M-orthonormal) and within themselves: Cholesky-QR
    done twice on the Gram GM.  Returns the new coefficients, or None when the block is numerically dependent and allow_drop is
    False; with allow_drop the dependent directions are dropped instead (eigen-decomposition of the projected Gram)."""
    d = np.sqrt(np.maximum(np.einsum("ij,ik,kj->j", V, GM, V), 0.0))
    if np.any(d == 0.0) and not allow_drop:
        return None
    V = V[:, d > 0] / d[d > 0]
    for sweep in range(2):
        if Q.shape[1]:
            V = V - Q @ (Q.T @ GM @ V)
        H = V.T @ GM @ V
        H = 0.5 * (H + H.T)
        try:
            L = np.linalg.cholesky(H)
            ok = sweep == 1 or pivot == 0.0 or np.diag(L).min() >= pivot
        except np.linalg.LinAlgError:
            ok = False
        if not ok:
            if not allow_drop:
                return None
            e, U = np.linalg.eigh(H)
            keep = e > DEPENDENT_PIVOT ** 2 * max(e.max(), 1.0)
            V = V @ (U[:, keep] / np.sqrt(e[keep]))
            continue
        V = np.linalg.solve(L, V.T).T      # V L^-T
    return V


def _rayleigh_ritz(GK, GM, blocks, m):
    """Basis coefficients T (S -> M-orthonormal basis, block by block) and the m lowest Ritz pairs of (T^T GK T, T^T GM T).
    `blocks`: list of (column indices, role) with role 'x', 'w' or 'p'.  Returns (lam, Z over S, Z restricted to the W/P part,
    P dropped?)."""
    dim = GK.shape[0]
    GK, GM = 0.5 * (GK + GK.T), 0.5 * (GM + GM.T)
    Q = np.zeros((dim, 0))
    nx = 0
    dropped = False
    for cols, role in blocks:
        if len(cols) == 0:
            continue
        V = np.zeros((dim, len(cols)))
        V[cols, np.arange(len(cols))] = 1.0
        V = _orthonormalise(GM, V, Q, allow_drop=role != "p", pivot=0.0 if role == "x" else DEPENDENT_PIVOT)
        if V is None:
            dropped = True
            continue
        Q = np.concatenate([Q, V], axis=1)
        if role == "x":
            nx = Q.shape[1]
    A, B = Q.T @ GK @ Q, Q.T @ GM @ Q
    L = np.linalg.cholesky(0.5 * (B + B.T))   # B = I up to rounding: Q is M-orthonormal
    Li = np.linalg.inv(L)
    lam, Y = np.linalg.eigh(0.5 * (Li @ A @ Li.T + (Li @ A @ Li.T).T))
    Z = Li.T @ Y[:, :m]
    return lam[:m], Q @ Z, Q[:, nx:] @ Z[nx:], dropped


# ------------------------------------------------------------------------------------------------------------------ driver

def lobpcg(be, num_eigs, tol=1e-8, max_iter=2000, X0=None):
    """Lowest num_eigs eigenpairs of the masked pencil held by the backend `be`.
    Returns (lam [num_eigs] ascending (numpy), S (the backend's [n, 3m] basis buffer; columns :num_eigs are the M-orthonormal
    modes), info dict)."""
    n, m = be.n, block_width(num_eigs)
    w3 = 3 * m
    maskh = be.mask_host().astype(np.float64)
    X0h = start_block(n, m, X0) * maskh[:, None]
    t0 = time.perf_counter()
    # initial Rayleigh-Ritz on the start block; a numerically dependent block keeps its independent Ritz vectors and is
    # refilled from the generator once
    KXt, MXt = be.zeros(n, m), be.zeros(n, m)
    buf = be.zeros(1, 2 * w3 * w3 + 2 * m).reshape(-1)
    for refill in range(2):
        Xt = be.upload(X0h)
        be.spmm(Xt, 0, m, KXt, MXt)
        be.gram(Xt, KXt, m, buf[:m * m])
        be.gram(Xt, MXt, m, buf[w3 * w3:w3 * w3 + m * m])
        h = be.host(buf)
        lam, Z, _, _ = _rayleigh_ritz(h[:m * m].reshape(m, m), h[w3 * w3:w3 * w3 + m * m].reshape(m, m), [(np.arange(m), "x")], m)
        r = Z.shape[1]
        if r == m or refill:
            break
        Xr = be.zeros(n, r)
        be.combine(Xt, m, Z, Xr, 0)
        fill = np.random.default_rng(START_SEED + 1).standard_normal((n, m - r)) * maskh[:, None]
        X0h = np.concatenate([be.host(Xr), fill], axis=1)
    S, KS, MS = (be.zeros(n, w3) for _ in range(3))
    nxt = [be.zeros(n, w3) for _ in range(3)]
    for src, dst in ((Xt, S), (KXt, KS), (MXt, MS)):
        be.combine(src, m, Z, dst, 0)
    del Xt, KXt, MXt
    active = list(range(m))
    act_dev = be.active_list(active)
    has_p, restarts, it = False, 0, 0
    norms = buf[2 * w3 * w3:]
    status = "maxiter"
    while True:
        na = len(active)
        be.residual(S, KS, MS, m, lam, act_dev, na, S, m, norms)
        if it == max_iter:
            h = be.host(buf)
        else:
            if na:
                be.spmm(S, m, na, KS, MS)
            k = w3 if has_p else 2 * m
            be.gram(S, KS, k, buf[:k * k])
            be.gram(S, MS, k, buf[w3 * w3:w3 * w3 + k * k])
            h = be.host(buf)
        rr, xx = h[2 * w3 * w3:2 * w3 * w3 + m], h[2 * w3 * w3 + m:2 * w3 * w3 + 2 * m]
        res = np.sqrt(np.maximum(rr, 0.0)) / ((be.norm_K + np.abs(lam) * be.norm_M) * np.sqrt(np.maximum(xx, 1e-300)))
        if np.all(res[:num_eigs] <= tol):
            status = "converged"
            break
        if it == max_iter:
            break
        blocks = [(np.arange(m), "x"), (m + np.arange(na), "w")]
        if has_p:
            blocks.append((2 * m + np.asarray(active, dtype=np.int64), "p"))
        GK, GM = h[:k * k].reshape(k, k), h[w3 * w3:w3 * w3 + k * k].reshape(k, k)
        lam, CX, CP, dropped = _rayleigh_ritz(GK, GM, blocks, m)
        restarts += int(dropped)
        S2, KS2, MS2 = nxt
        for src, dst in ((S, S2), (KS, KS2), (MS, MS2)):   # the new X and P and their products: no SpMM repeated
            be.combine(src, k, CX, dst, 0)
            be.combine(src, k, CP, dst, 2 * m)
        nxt = [S, KS, MS]
        S, KS, MS = S2, KS2, MS2
        has_p = True
        still = [j for j in active if res[j] > tol]
        if still != active:
            active = still
            act_dev = be.active_list(active) if active else None
        it += 1
    loop_ms = (time.perf_counter() - t0) * 1e3
    info = {"iterations": it, "status": status, "residuals": res[:num_eigs].copy(), "restarts": restarts,
            "freq_hz": np.sqrt(np.maximum(lam[:num_eigs], 0.0)) / (2 * np.pi), "loop_ms": loop_ms}
    return np.asarray(lam[:num_eigs]).copy(), S, info
