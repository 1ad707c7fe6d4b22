"""Smoothed-aggregation algebraic multigrid (Vanek, Mandel & Brezina 1996) for 3-dof solid operators: the V-cycle of
femb200/multigrid.py on a hierarchy built from the assembled operator and the node coordinates alone, so any solid mesh gets it.

Every level is a square 3x3 block-CSR operator.  The near-nullspace is the six rigid-body modes.  Level l+1 comes from level l in
five device steps (csrc/amg.cu):
  aggregate   distance-2 maximal independent set of the node graph (every pattern connection, no strength threshold); roots take
              their neighbours, the rest join the neighbouring aggregate with the lowest id; nodes with all dofs fixed stay out
  tentative   per aggregate a, CholQR2 of its near-nullspace B_a [3 n_a, 6] = [I3 | -skew(x_i - c_a)] with the rotation columns
              scaled by 1 / aggregate diameter; coarser levels carry the global modes down and re-centre them the same way (their
              pseudo-nodes sit at the centroids of the aggregates they came from).  B_a = Q_a R_a: Q_a gives two 3x3 blocks per
              fine node, at coarse pseudo-nodes 2a (translations) and 2a+1 (rotations); R_a, mapped back to the global modes, is
              the coarse near-nullspace.
              A column whose pivot is <= DROP_PIVOT (relative) is dropped and its coarse dof masked (one free node: no rotations).
  lam         lam ~ rho(D^-1 A) by POWER_ITERS power steps from a fixed seed (femb_spmv_bsr3); omega = 4 / (3 lam)
  smooth      P = S P_tent with S = mask (I - omega D^-1 A) formed on A's pattern (femb_bsr3_spgemm), R = P^T (femb_bsr3_transpose)
  Galerkin    A_c = R (A P) (two femb_bsr3_spgemm)
Coarsening stops when a level has at most `coarse_dofs` free dofs (COARSE_DOFS by default), or when the next level would keep more
than half of them; the last level is factorised densely (Hierarchy._factor), so it may hold at most multigrid.MAX_COARSE_DOFS.
Every step sums in a fixed order: a repeated setup is bit-identical.  In the cycle the transfers are femb_mg_transfer_bsr3.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch

from . import multigrid, ops
from ._lib import check, lib
from .modes import _p

COARSE_DOFS = 2000        # free dofs at which coarsening stops: the dense factor of 2,000 dofs is 32 MB and a few ms to build
DROP_PIVOT = 1e-10        # a CholQR pivot below this times the largest Gram diagonal drops its near-nullspace column
POWER_ITERS = 15          # power steps for the largest eigenvalue of D^-1 A
POWER_SEED = 20261022


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def aggregate(A, mask):
    """(agg int32 [nb], number of aggregates) of the node graph of A (femb_amg_aggregate)."""
    agg = torch.empty(A.nb, device=A.dev, dtype=torch.int32)
    n = C.c_int64()
    with torch.cuda.device(A.dev):
        check(lib.femb_amg_aggregate(A.nb, _p(A.brow), _p(A.bcol), _p(mask), _p(agg), C.byref(n), _stream(A.dev)), "femb_amg_aggregate")
    return agg, n.value


def tentative(agg, n_agg, mask, coords, B=None):
    """(P_tent as ops.Bsr3 with n_fine block rows, coarse near-nullspace [6 n_agg, 6], coarse mask uint8 [6 n_agg], coarse coordinates
    [2 n_agg, 3]) (femb_amg_tentative).  B None: the finest level (rigid-body modes of coords)."""
    dev = agg.device
    nb = agg.numel()
    nin = int((agg >= 0).sum())
    prow = torch.empty(nb + 1, device=dev, dtype=torch.int32)
    pcol = torch.empty(2 * nin, device=dev, dtype=torch.int32)
    pval = torch.empty((2 * nin, 3, 3), device=dev, dtype=torch.float64)
    Bc = torch.empty((6 * n_agg, 6), device=dev, dtype=torch.float64)
    mask_c = torch.empty(6 * n_agg, device=dev, dtype=torch.uint8)
    coords_c = torch.empty((2 * n_agg, 3), device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        check(lib.femb_amg_tentative(nb, n_agg, _p(agg), _p(mask), _p(coords), _p(B), DROP_PIVOT, _p(prow), _p(pcol), _p(pval), _p(Bc),
                                     _p(mask_c), _p(coords_c), _stream(dev)), "femb_amg_tentative")
    return ops.Bsr3(prow, pcol, pval), Bc, mask_c, coords_c


def spgemm(X, Y):
    """C = X Y for 3x3 block-CSR (ops.Bsr3; X's block columns index Y's block rows) (femb_bsr3_spgemm, symbolic then numeric)."""
    dev = X.dev
    crow = torch.empty(X.nb + 1, device=dev, dtype=torch.int32)
    nnz = C.c_int64()
    with torch.cuda.device(dev):
        check(lib.femb_bsr3_spgemm(X.nb, _p(X.brow), _p(X.bcol), None, _p(Y.brow), _p(Y.bcol), None, _p(crow), None, None, C.byref(nnz),
                                   _stream(dev)), "femb_bsr3_spgemm")
        ccol = torch.empty(nnz.value, device=dev, dtype=torch.int32)
        cval = torch.empty((nnz.value, 3, 3), device=dev, dtype=torch.float64)
        check(lib.femb_bsr3_spgemm(X.nb, _p(X.brow), _p(X.bcol), _p(X.bval), _p(Y.brow), _p(Y.bcol), _p(Y.bval), _p(crow), _p(ccol), _p(cval),
                                   None, _stream(dev)), "femb_bsr3_spgemm")
    return ops.Bsr3(crow, ccol, cval)


def transpose(P, n_cols):
    """R = P^T with transposed blocks (femb_bsr3_transpose)."""
    dev = P.dev
    rrow = torch.empty(n_cols + 1, device=dev, dtype=torch.int32)
    rcol = torch.empty(P.nnzb, device=dev, dtype=torch.int32)
    rval = torch.empty((P.nnzb, 3, 3), device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        check(lib.femb_bsr3_transpose(P.nb, n_cols, P.nnzb, _p(P.brow), _p(P.bcol), _p(P.bval), _p(rrow), _p(rcol), _p(rval), _stream(dev)),
              "femb_bsr3_transpose")
    return ops.Bsr3(rrow, rcol, rval)


def spectral_radius(A, dinv):
    """lam ~ rho(D^-1 A) by POWER_ITERS power steps from a fixed seed (masked dofs: dinv = 0)."""
    x = torch.from_numpy(np.random.default_rng(POWER_SEED).standard_normal(3 * A.nb)).to(A.dev) * (dinv != 0)
    lam = 0.0
    for _ in range(POWER_ITERS):
        nx = float(torch.linalg.vector_norm(x))
        if nx == 0.0:
            return 0.0
        x = dinv * A.spmv(x / nx)
        lam = float(torch.linalg.vector_norm(x))
    return lam


def smoother_matrix(A, mask, dinv, omega):
    """S = mask (I - omega D^-1 A) on A's pattern (A's diagonal blocks are in the pattern)."""
    rows = torch.repeat_interleave(torch.arange(A.nb, device=A.dev), (A.brow[1:] - A.brow[:-1]).long())
    sval = -omega * dinv.reshape(-1, 3)[rows][:, :, None] * A.bval
    diag = A.bcol.long() == rows
    sval[diag] += torch.diag_embed(mask.reshape(-1, 3)[rows[diag]].to(torch.float64))
    return ops.Bsr3(A.brow, A.bcol, sval)


class Level:
    """One level of the algebraic hierarchy: A, mask, dinv, the cycle buffers, and (above the coarsest) P, R to the level below."""

    def __init__(self, A, mask):
        self.A, self.mask = A, mask
        self.nodes, self.n, self.tets = A.nb, 3 * A.nb, None
        self.free = int(mask.sum())
        self.dinv = A.jacobi(mask)
        self.P = self.R = None
        self.K = self.M = None
        self.b, self.x, self.y, self.t = (multigrid.level_buffer(self.n, A.dev) for _ in range(4))

    def restrict(self, coarse, na, X, stream):
        """coarse.b[:, :na] = coarse.mask (R X) (femb_mg_transfer_bsr3)."""
        _block_transfer(self.R, coarse.nodes, self.nodes, coarse.mask, na, X, coarse.b, False, stream)

    def prolong(self, coarse, na, Xc, Y, stream):
        """Y[:, :na] += mask (P Xc) (femb_mg_transfer_bsr3)."""
        _block_transfer(self.P, self.nodes, coarse.nodes, self.mask, na, Xc, Y, True, stream)


def _block_transfer(T, n_out, n_in, mask_out, na, X, Y, accumulate, stream):
    W = multigrid.WIDTH
    with torch.cuda.device(X.device):
        check(lib.femb_mg_transfer_bsr3(n_out, n_in, T.nnzb, _p(T.brow), _p(T.bcol), _p(T.bval), _p(mask_out), na, _p(X), W, int(accumulate),
                                        _p(Y), W, stream), "femb_mg_transfer_bsr3")


class AmgHierarchy(multigrid.Hierarchy):
    """Smoothed-aggregation hierarchy of A (ops.Bsr3, the operator the cycle approximates the inverse of) with dof mask `mask` (uint8,
    0 = fixed) and node coordinates `coords` [N, 3].  K, M: the pencil kept on the finest level for LOBPCG (multigrid.MultilevelBackend).
    The cycle, apply and the backends are those of multigrid.Hierarchy.  Raises ValueError when coarsening stalls above
    multigrid.MAX_COARSE_DOFS free dofs, or when the coarsest operator is singular on its free dofs (a free-free model needs a shift).
    A Galerkin product row holds at most 2,048 blocks (femb_bsr3_spgemm's per-row capacity; solid meshes stay far below it): a wider
    row raises FembError, and a smaller `coarse_dofs` does not help, since the rows grow with coarsening."""

    def __init__(self, A, mask, coords, K=None, M=None, coarse_dofs=COARSE_DOFS):
        dev = self.dev = A.dev
        self.shift = None
        self.stream = _stream(dev)
        coords = torch.as_tensor(coords).to(dev, torch.float64).contiguous()
        if coords.shape != (A.nb, 3):
            raise ValueError(f"coords must be [{A.nb}, 3], got {tuple(coords.shape)}")
        self.setup_ms = dict.fromkeys(("aggregation", "tentative", "lambda", "spgemm", "factor"), 0.0)
        t = [time.perf_counter()]

        def lap(key):
            torch.cuda.synchronize(dev)
            now = time.perf_counter()
            self.setup_ms[key] += 1e3 * (now - t[0])
            t[0] = now

        fine = Level(A, mask)
        fine.K, fine.M = K, M
        levels, B = [fine], None
        while levels[-1].free > coarse_dofs:
            lv = levels[-1]
            agg, n_agg = aggregate(lv.A, lv.mask)
            lap("aggregation")
            Pt, Bc, mask_c, coords_c = tentative(agg, n_agg, lv.mask, coords, B)
            lap("tentative")
            if 2 * int(mask_c.sum()) > lv.free:   # coarsening stalled: this level is the coarsest
                break
            omega = 4.0 / (3.0 * spectral_radius(lv.A, lv.dinv))
            lap("lambda")
            P = spgemm(smoother_matrix(lv.A, lv.mask, lv.dinv, omega), Pt)
            R = transpose(P, 2 * n_agg)
            Ac = spgemm(R, spgemm(lv.A, P))
            lap("spgemm")
            lv.P, lv.R = P, R
            levels.append(Level(Ac, mask_c))
            B, coords = Bc, coords_c
        self.L = levels[::-1]
        if self.L[0].free > multigrid.MAX_COARSE_DOFS:
            raise ValueError(f"algebraic coarsening stalled at {self.L[0].free} free dofs; the dense coarsest level allows at most "
                             f"{multigrid.MAX_COARSE_DOFS}")
        self._factor(self.L[0])
        lap("factor")

    def describe(self):
        """Per level (coarsest first) nodes, dofs, free dofs and nnzb, the operator complexity (sum of nnzb over the finest level's)
        and the setup time split in ms."""
        levels = [{"nodes": lv.nodes, "dofs": lv.n, "free_dofs": lv.free, "nnzb": lv.A.nnzb} for lv in self.L]
        return {"levels": levels, "operator_complexity": sum(lv.A.nnzb for lv in self.L) / self.L[-1].A.nnzb,
                "setup_ms": dict(self.setup_ms)}
