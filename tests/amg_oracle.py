"""Numpy restatement of the smoothed-aggregation hierarchy of femb200/amg.py and its kernels (csrc/amg.cu, femb_mg_transfer_bsr3)
-- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Block operators are (brow, bcol, bval [nnzb, 3, 3]) triplets; `dof(T, n_cols)` turns one into a scipy CSR over dofs.  `NumpyAmg`
builds the hierarchy and runs the V(SMOOTH, SMOOTH) cycle of femb200.multigrid.Hierarchy on it; `NumpyAmgBackend` is the LOBPCG
backend of oracle/modes_oracle.py with that cycle in its residual step, so amg_lowest_modes' algorithm runs without a GPU.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl
import scipy.sparse as sp

from oracle import modes_oracle as MO

SMOOTH, OMEGA = 2, 0.5
COARSE_DOFS, DROP_PIVOT, POWER_ITERS, POWER_SEED = 2000, 1e-10, 15, 20261022
MAX_COARSE_DOFS, SINGULAR_PIVOT = 30000, 1e-12


def node_hash(i):
    x = np.asarray(i, dtype=np.uint64) & np.uint64(0xFFFFFFFF)
    m = np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7FEB352D)) & m
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846CA68B)) & m
    x ^= x >> np.uint64(16)
    return x


def edges(brow, bcol, incl):
    rows = np.repeat(np.arange(len(brow) - 1), np.diff(brow))
    keep = incl[rows] & incl[bcol]
    return rows[keep], np.asarray(bcol)[keep].astype(np.int64)


def mis_roots(brow, bcol, mask):
    """(included-node flags, root ids in increasing order) of the distance-2 independent set."""
    nb = len(brow) - 1
    incl = np.asarray(mask).reshape(nb, 3).any(axis=1) if mask is not None else np.ones(nb, dtype=bool)
    r, c = edges(brow, bcol, incl)
    ids = np.arange(nb, dtype=np.uint64)
    base = ((node_hash(ids) >> np.uint64(1)) << np.uint64(31)) | ids
    st = np.where(incl, 1, -1)
    while True:
        key = (np.maximum(st, 0).astype(np.uint64) << np.uint64(62)) | base
        t1 = key.copy()
        np.maximum.at(t1, r, key[c])
        t2 = t1.copy()
        np.maximum.at(t2, r, t1[c])
        und = st == 1
        root = und & ((t2 & np.uint64(0x7FFFFFFF)) == ids)
        out = und & ~root & ((t2 >> np.uint64(62)) == 2)
        st[root], st[out] = 2, 0
        if not (st == 1).any():
            break
    return incl, np.nonzero(st == 2)[0]


def aggregate(brow, bcol, mask):
    """femb_amg_aggregate: (agg int32 [nb], n_agg)."""
    nb = len(brow) - 1
    incl, roots = mis_roots(brow, bcol, mask)
    r, c = edges(brow, bcol, incl)
    is_root = np.zeros(nb, dtype=bool)
    is_root[roots] = True
    rank = np.cumsum(is_root) - is_root
    agg1 = np.where(is_root, rank, -1)
    hit = is_root[c] & ~is_root[r]
    agg1[r[hit]] = rank[c[hit]]
    agg = agg1.copy()
    cand = np.full(nb, np.iinfo(np.int64).max)
    ok = (agg1[c] >= 0) & (agg1[r] < 0)
    np.minimum.at(cand, r[ok], agg1[c[ok]])
    left = (agg1 < 0) & incl
    agg[left] = cand[left]
    return agg.astype(np.int32), int(is_root.sum())


def chol_drop(G, drop):
    L = np.zeros((6, 6))
    kept = np.ones(6, dtype=bool)
    gmax = np.diag(G).max()
    for k in range(6):
        d = G[k, k] - L[k, :k] @ L[k, :k]
        if not d > drop * gmax:
            kept[k] = False
            continue
        L[k, k] = np.sqrt(d)
        L[k + 1:, k] = (G[k + 1:, k] - L[k + 1:, :k] @ L[k, :k]) / L[k, k]
    return L, kept


def solve_rows(B, L, kept):
    Q = np.zeros_like(B)
    for k in range(6):
        if kept[k]:
            Q[:, k] = (B[:, k] - Q[:, :k] @ L[k, :k]) / L[k, k]
    return Q


def rigid_rows(x, c, s):
    """[3 n, 6] rows [I3 | e_k x (x - c) s] of the nodes x [n, 3]."""
    r = (x - c) * s
    n = x.shape[0]
    B = np.zeros((n, 3, 6))
    for d in range(3):
        B[:, d, d] = 1.0
    B[:, 1, 3], B[:, 2, 3] = -r[:, 2], r[:, 1]
    B[:, 0, 4], B[:, 2, 4] = r[:, 2], -r[:, 0]
    B[:, 0, 5], B[:, 1, 5] = -r[:, 1], r[:, 0]
    return B.reshape(3 * n, 6)


def tentative(agg, n_agg, mask, coords, B=None, drop=DROP_PIVOT):
    """femb_amg_tentative: ((prow, pcol, pval), Bc [6 n_agg, 6], mask_c uint8 [6 n_agg], coords_c [2 n_agg, 3])."""
    nb = agg.size
    f = np.asarray(mask, dtype=np.float64).reshape(nb, 3) if mask is not None else np.ones((nb, 3))
    prow = np.concatenate([[0], 2 * np.cumsum(agg >= 0)]).astype(np.int32)
    pcol = np.empty(prow[-1], dtype=np.int32)
    pval = np.empty((prow[-1], 3, 3))
    Bc = np.zeros((6 * n_agg, 6))
    mask_c = np.zeros(6 * n_agg, dtype=np.uint8)
    coords_c = np.zeros((2 * n_agg, 3))
    order = np.argsort(agg, kind="stable")
    order = order[agg[order] >= 0]
    starts = np.searchsorted(agg[order], np.arange(n_agg + 1))
    for a in range(n_agg):
        nodes = order[starts[a]:starts[a + 1]]
        x = coords[nodes]
        cen = x.sum(axis=0) / nodes.size
        rmax = np.sqrt(((x - cen) ** 2).sum(axis=1)).max()
        s = 1.0 / (2.0 * rmax) if rmax > 0 else 1.0
        T = np.eye(6)                                            # local -> global rigid-body columns
        T[3:, 3:] /= s
        T[:3, 3:] = rigid_rows(cen[None, :], np.zeros(3), 1.0)[:, 3:]
        if B is None:
            Ba = rigid_rows(x, cen, s)
        else:                                                    # global modes carried down, re-centred: B T^-1
            Ba = B.reshape(nb, 3, 6)[nodes].reshape(-1, 6) @ np.linalg.inv(T)
        Ba *= f[nodes].reshape(-1, 1)
        L1, k1 = chol_drop(Ba.T @ Ba, drop)
        Q1 = solve_rows(Ba, L1, k1)
        L2, k2 = chol_drop(Q1.T @ Q1, drop)
        kept = k1 & k2
        Q = solve_rows(Q1, L2, k2) * kept
        Rm = ((L2.T @ L1.T) * kept[:, None]) @ T
        Qn = Q.reshape(-1, 3, 6)
        pos = prow[nodes]
        pval[pos], pval[pos + 1] = Qn[:, :, :3], Qn[:, :, 3:]
        pcol[pos], pcol[pos + 1] = 2 * a, 2 * a + 1
        Bc[6 * a:6 * a + 6] = Rm
        mask_c[6 * a:6 * a + 6] = kept
        coords_c[2 * a:2 * a + 2] = cen
    return (prow, pcol, pval), Bc, mask_c, coords_c


def dof(T, n_cols):
    """scipy CSR over dofs of a block triplet with n_cols block columns."""
    brow, bcol, bval = (np.asarray(a) for a in T)
    return sp.bsr_matrix((bval, bcol, brow), shape=(3 * (len(brow) - 1), 3 * n_cols)).tocsr()


def pattern(T, n_cols):
    brow, bcol, _ = T
    return sp.csr_matrix((np.ones(len(bcol)), np.asarray(bcol), np.asarray(brow)), shape=(len(brow) - 1, n_cols))


def blocks(D, pat):
    """Block triplet of the dof-level matrix D on the block pattern `pat` (scipy CSR, sorted)."""
    pat = pat.tocsr()
    pat.sort_indices()
    rows = np.repeat(np.arange(pat.shape[0]), np.diff(pat.indptr))
    d = np.arange(3)
    Dd = D.tocsr()
    ri, ci = np.broadcast_arrays(3 * rows[:, None, None] + d[:, None], 3 * pat.indices[:, None, None] + d[None, :])
    vals = np.asarray(Dd[ri.reshape(-1), ci.reshape(-1)]).reshape(-1, 3, 3)
    return pat.indptr.astype(np.int32), pat.indices.astype(np.int32), vals


def spgemm(X, Y, n_cols_x, n_cols_y):
    """femb_bsr3_spgemm: the block pattern of X Y (every structural product) and its values."""
    pat = (pattern(X, n_cols_x) @ pattern(Y, n_cols_y))
    return blocks(dof(X, n_cols_x) @ dof(Y, n_cols_y), pat)


def transpose(P, n_cols):
    return blocks(dof(P, n_cols).T, pattern(P, n_cols).T)


def spectral_radius(A, dinv):
    x = np.random.default_rng(POWER_SEED).standard_normal(A.shape[0]) * (dinv != 0)
    lam = 0.0
    for _ in range(POWER_ITERS):
        nx = np.linalg.norm(x)
        if nx == 0.0:
            return 0.0
        x = dinv * (A @ (x / nx))
        lam = np.linalg.norm(x)
    return lam


def jacobi(A, mask):
    d = A.diagonal()
    return np.where((mask != 0) & (d != 0), 1.0 / np.where(d != 0, d, 1.0), 0.0)


def smoother(T, mask, dinv, omega):
    brow, bcol, bval = T
    rows = np.repeat(np.arange(len(brow) - 1), np.diff(brow))
    sval = -omega * dinv.reshape(-1, 3)[rows][:, :, None] * bval
    diag = np.asarray(bcol) == rows
    sval[diag] += mask.reshape(-1, 3)[rows[diag]][:, :, None] * np.eye(3)
    return brow, bcol, sval


class NumpyAmg:
    """The hierarchy of femb200.amg.AmgHierarchy (finest first in `levels`, as dicts with T: block triplet, A: dof CSR, mask, dinv,
    agg, P, R block triplets) and its V-cycle."""

    def __init__(self, T, mask, coords, coarse_dofs=COARSE_DOFS):
        lv = self._level(T, mask)
        self.levels, B = [lv], None
        while int(lv["mask"].sum()) > coarse_dofs:
            agg, n_agg = aggregate(T[0], T[1], lv["mask"])
            Pt, Bc, mask_c, coords_c = tentative(agg, n_agg, lv["mask"], coords, B)
            lv["agg"], lv["Pt"], lv["Bc"] = agg, Pt, Bc
            if 2 * int(mask_c.sum()) > int(lv["mask"].sum()):
                break
            omega = 4.0 / (3.0 * spectral_radius(lv["A"], lv["dinv"]))
            nc = 2 * n_agg
            P = spgemm(smoother(T, lv["mask"], lv["dinv"], omega), Pt, lv["nodes"], nc)
            R = transpose(P, nc)
            T = spgemm(R, spgemm(T, P, lv["nodes"], nc), lv["nodes"], nc)
            lv["P"], lv["R"], lv["omega"] = P, R, omega
            lv = self._level(T, mask_c)
            self.levels.append(lv)
            B, coords = Bc, coords_c
        c = self.levels[-1]
        self.free0 = c["mask"] != 0
        A0 = c["A"].toarray()[np.ix_(self.free0, self.free0)]
        try:
            self.chol0 = sl.cho_factor(A0, lower=True)
        except np.linalg.LinAlgError:
            self.chol0 = None
        if self.chol0 is None or (A0.size and np.diag(self.chol0[0]).min() ** 2 < SINGULAR_PIVOT * np.diag(A0).max()):
            raise ValueError("the coarse operator K + shift M is singular on the free dofs: pass shift > 0")

    @staticmethod
    def _level(T, mask):
        nodes = len(T[0]) - 1
        A = dof(T, nodes)
        mask = np.asarray(mask, dtype=np.uint8)
        return {"T": T, "A": A, "mask": mask, "dinv": jacobi(A, mask), "nodes": nodes}

    def smooth(self, lv, b, x):
        f = lv["mask"][:, None].astype(np.float64)
        t = f * (b - (lv["A"] @ (f * x) if x is not None else 0.0))
        return (x if x is not None else 0.0) + OMEGA * lv["dinv"][:, None] * t, t

    def cycle(self, k, b):
        if k == len(self.levels) - 1:
            x = np.zeros_like(b)
            x[self.free0] = sl.cho_solve(self.chol0, b[self.free0])
            return x
        lv, cl = self.levels[k], self.levels[k + 1]
        x, _ = self.smooth(lv, b, None)
        for _ in range(SMOOTH - 1):
            x, _ = self.smooth(lv, b, x)
        _, t = self.smooth(lv, b, x)
        xc = self.cycle(k + 1, transfer(lv["R"], cl["mask"], t, lv["nodes"]))
        x = transfer(lv["P"], lv["mask"], xc, cl["nodes"], x)
        for _ in range(SMOOTH):
            x, _ = self.smooth(lv, b, x)
        return x

    def apply(self, B):
        return self.cycle(0, np.asarray(B, dtype=np.float64))


def transfer(T, mask_out, X, n_in, Y=None):
    """femb_mg_transfer_bsr3: Y (+)= mask_out (T X)."""
    out = (dof(T, n_in) @ X) * np.asarray(mask_out, dtype=np.float64)[:, None]
    return out if Y is None else Y + out


class NumpyAmgBackend(MO.NumpyBackend):
    """MO.NumpyBackend (pencil kval, mval) whose residual step preconditions with the AMG V-cycle of A = K + shift M."""

    def __init__(self, brow, bcol, kval, mval, mask, coords, shift=0.0, coarse_dofs=COARSE_DOFS):
        super().__init__(brow, bcol, kval, mval, mask)
        self.H = NumpyAmg((brow, bcol, kval + shift * mval), self.mask, coords, coarse_dofs)

    def residual(self, X, KX, MX, m, lam, active, na, W, c0, norms):
        R = KX[:, :m] - MX[:, :m] * np.asarray(lam, dtype=np.float64)[None, :m]
        norms[:m] = (R * R).sum(axis=0)
        norms[m:2 * m] = (X[:, :m] * X[:, :m]).sum(axis=0)
        if na:
            W[:, c0:c0 + na] = self.H.apply(self.mask[:, None] * R[:, np.asarray(active)[:na]])
