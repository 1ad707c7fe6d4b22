"""Numpy restatement of the multigrid preconditioner of subdivided_lowest_modes (femb200/multigrid.py and the kernels
femb_mg_smooth_bsr3 / femb_mg_transfer of csrc/modes.cu) -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

`NumpyMultilevelBackend` is the LOBPCG backend of oracle/modes_oracle.py with the V-cycle in its residual step, so the whole
algorithm (femb200.modes.lobpcg) runs on a CPU-only machine.  A hierarchy is a list of level dicts, coarsest first:
brow, bcol, aval [nnzb, 3, 3] (A_s = K + shift M), mask uint8 [3 N]; every refined level also P and R as node-level CSR
triplets (crow, col, val).  `numpy_hierarchy` builds one with a numpy refine_once; on the GPU `from_device` hands the arrays of a
device-built femb200.multigrid.Hierarchy to the same code.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl
import scipy.sparse as sp

from oracle import fem_oracle as O
from oracle import modes_oracle as MO

SMOOTH, OMEGA = 2, 0.5
SINGULAR_PIVOT = 1e-12


# ------------------------------------------------------------------------------------------------------- kernel restatements

def smooth(A, mask, dinv, omega, R, X_in):
    """femb_mg_smooth_bsr3: t = mask (R - A (mask X_in)), X_out = X_in + omega dinv t (X_in None = 0).  Returns (X_out, t)."""
    f = mask[:, None].astype(np.float64)
    AX = A @ (f * X_in) if X_in is not None else 0.0
    t = f * (R - AX)
    return (X_in if X_in is not None else 0.0) + omega * dinv[:, None] * t, t


def transfer(S, mask_out, X, Y=None):
    """femb_mg_transfer: Y[3i+d] (+)= mask_out[3i+d] sum_k S_ik X[3k+d] (S node-level scipy CSR)."""
    k = X.shape[1]
    out = (S @ X.reshape(S.shape[1], 3 * k)).reshape(3 * S.shape[0], k) * mask_out[:, None].astype(np.float64)
    return out if Y is None else Y + out


def csr(triplet, shape):
    crow, col, val = (np.asarray(a) for a in triplet)
    return sp.csr_matrix((val, col, crow), shape=shape)


# ------------------------------------------------------------------------------------------------------------- hierarchy

def refine_once(coords, tets):
    """fem_oracle.c3d4_to_c3d10 + the 8-child split: (coords', tets', parents [N'-N, 2])."""
    N = coords.shape[0]
    c10, e10 = O.c3d4_to_c3d10(coords, tets)
    parents = np.empty((c10.shape[0] - N, 2), dtype=np.int64)
    parents[e10[:, 4:].reshape(-1) - N] = e10[:, np.array(O.P2_MID_EDGES)].reshape(-1, 2)
    return c10, O.to_c3d4(e10), parents


def prolongation(parents, n_coarse):
    nm = parents.shape[0]
    rows = np.concatenate([np.arange(n_coarse), n_coarse + np.repeat(np.arange(nm), 2)])
    cols = np.concatenate([np.arange(n_coarse), np.sort(parents, axis=1).reshape(-1)])
    vals = np.concatenate([np.ones(n_coarse), np.full(2 * nm, 0.5)])
    P = sp.csr_matrix((vals, (rows, cols)), shape=(n_coarse + nm, n_coarse))
    R = P.T.tocsr()
    R.sort_indices()
    return (P.indptr, P.indices, P.data), (R.indptr, R.indices, R.data)


def numpy_hierarchy(coords, tets, levels, fixed_fn, E, nu, rho, shift=0.0):
    """Level dicts of a coarse C3D4 mesh refined `levels` times, plus the finest K and M block values and mesh:
    (levels, kval, mval, coords, tets)."""
    coords, tets = np.asarray(coords, dtype=np.float64), np.asarray(tets, dtype=np.int64)
    out = []
    parents = None
    for k in range(levels + 1):
        if k:
            coords, tets, parents = refine_once(coords, tets)
        N = coords.shape[0]
        pat = MO.node_pattern(tets, N)
        kval = MO.assemble_bsr3(O.c3d4_K(coords, tets, E, nu), tets, N, pat)
        mval = MO.assemble_bsr3(O.c3d4_mass(coords, tets, rho), tets, N, pat)
        lv = {"brow": pat[0], "bcol": pat[1], "aval": kval + shift * mval, "mask": MO.dof_mask(N, fixed_fn(coords))}
        if parents is not None:
            lv["P"], lv["R"] = prolongation(parents, N - parents.shape[0])
        out.append(lv)
    return out, kval, mval, coords, tets


def from_device(H):
    """The level dicts of a device-built femb200.multigrid.Hierarchy (same arrays, copied to the host)."""
    h = lambda t: t.cpu().numpy()  # noqa: E731
    out = []
    for lv in H.L:
        d = {"brow": h(lv.A.brow), "bcol": h(lv.A.bcol), "aval": h(lv.A.bval), "mask": h(lv.mask)}
        if lv.P is not None:
            d["P"], d["R"] = tuple(map(h, lv.P)), tuple(map(h, lv.R))
        out.append(d)
    return out


class NumpyHierarchy:
    """The V(SMOOTH, SMOOTH) cycle of femb200.multigrid.Hierarchy on level dicts."""

    def __init__(self, levels):
        self.L = []
        for k, lv in enumerate(levels):
            A = MO.bsr_matrix(lv["brow"], lv["bcol"], lv["aval"]).tocsr()
            mask = np.asarray(lv["mask"], dtype=np.uint8)
            d = A.diagonal()
            dinv = np.where((mask != 0) & (d != 0), 1.0 / np.where(d != 0, d, 1.0), 0.0)
            L = {"A": A, "mask": mask, "dinv": dinv, "nodes": A.shape[0] // 3}
            if k:
                nc = self.L[-1]["nodes"]
                L["P"], L["R"] = csr(lv["P"], (L["nodes"], nc)), csr(lv["R"], (nc, L["nodes"]))
            self.L.append(L)
        l0 = self.L[0]
        self.free0 = l0["mask"] != 0
        A0 = l0["A"].toarray()[np.ix_(self.free0, self.free0)]
        try:
            self.chol0 = sl.cho_factor(A0, lower=True)
        except np.linalg.LinAlgError:
            self.chol0 = None
        if self.chol0 is None or (A0.size and np.diag(self.chol0[0]).min() ** 2 < SINGULAR_PIVOT * np.diag(A0).max()):
            raise ValueError("the coarse operator K + shift M is singular on the free dofs: pass shift > 0")

    def cycle(self, l, b):
        if l == 0:
            x = np.zeros_like(b)
            x[self.free0] = sl.cho_solve(self.chol0, b[self.free0])
            return x
        lv, cl = self.L[l], self.L[l - 1]
        x, _ = smooth(lv["A"], lv["mask"], lv["dinv"], OMEGA, b, None)
        for _ in range(SMOOTH - 1):
            x, _ = smooth(lv["A"], lv["mask"], lv["dinv"], OMEGA, b, x)
        _, t = smooth(lv["A"], lv["mask"], lv["dinv"], OMEGA, b, x)
        xc = self.cycle(l - 1, transfer(lv["R"], cl["mask"], t))
        x = transfer(lv["P"], lv["mask"], xc, x)
        for _ in range(SMOOTH):
            x, _ = smooth(lv["A"], lv["mask"], lv["dinv"], OMEGA, b, x)
        return x

    def apply(self, B):
        return self.cycle(len(self.L) - 1, np.asarray(B, dtype=np.float64))


class NumpyMultilevelBackend(MO.NumpyBackend):
    """MO.NumpyBackend whose residual step preconditions with the V-cycle: W[:, c0+a] = V(mask r_active[a])."""

    def __init__(self, levels, kval, mval):
        top = levels[-1]
        super().__init__(top["brow"], top["bcol"], kval, mval, top["mask"])
        self.H = NumpyHierarchy(levels)

    def residual(self, X, KX, MX, m, lam, active, na, W, c0, norms):
        R = KX[:, :m] - MX[:, :m] * np.asarray(lam, dtype=np.float64)[None, :m]
        norms[:m] = (R * R).sum(axis=0)
        norms[m:2 * m] = (X[:, :m] * X[:, :m]).sum(axis=0)
        if na:
            W[:, c0:c0 + na] = self.H.apply(self.mask[:, None] * R[:, np.asarray(active)[:na]])
