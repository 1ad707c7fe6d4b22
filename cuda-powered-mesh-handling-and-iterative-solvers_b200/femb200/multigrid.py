"""Device V-cycle over a uniform-refinement hierarchy, the preconditioner of `subdivided_lowest_modes` (LOBPCG, femb200/modes.py).

The hierarchy is the one of the hybrid static solver (femb200/hybrid.py): a coarse C3D4 mesh refined `levels` times with
`hybrid.refine_once`, node-level prolongation P (a mid-edge node takes the mean of its parents) and restriction R = P^T.  Every
level holds A_s = K + shift M as 3x3 block-CSR (K itself when shift = 0), its dof mask and dinv = mask / diag(A_s).  The cycle is
V(SMOOTH, SMOOTH) with damped Jacobi (OMEGA) on the refined levels and a dense Cholesky solve of the free block of A_s on level 0,
so it approximates (K + shift M)^-1 on the free dofs; with clamped dofs shift = 0 is right, a free-free model needs shift > 0.

It works on LOBPCG's row-major multivectors: every level owns [3 N_l, 16] buffers (rhs, two ping-pong iterates, residual),
allocated once, and a cycle over na <= 16 columns is a fixed sequence of launches with no host synchronisation -- on the refined
levels two kernels of csrc/modes.cu, femb_mg_smooth_bsr3 (smoothing step / residual) and femb_mg_transfer (P and R), on level 0
a torch `cholesky_solve` (a library call is allowed for the coarse solve).  Per refined level and cycle: 2 SMOOTH - 1 + 1 passes
over A_s (the first smoothing step starts from x = 0 and reads no matrix), one restriction and one prolongation.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import hybrid, modes, ops
from ._lib import check, lib
from .modes import _p

SMOOTH = 2                 # damped-Jacobi steps before and after the coarse correction
OMEGA = 0.5                # Jacobi damping.  The 8-child split of refine_once (c3d10_to_c3d4) makes the largest eigenvalue of
                           # dinv A grow over the first refinements: on kuhn_cube(4) + 1, 2, 3 levels LOBPCG takes 13, 14, 14
                           # iterations at 0.5, 12, 13, 19 at 0.6 (hybrid.multilevel_solve's value) and fails at 0.7
MAX_COARSE_DOFS = 30000    # bound on the free dofs of level 0: its dense Cholesky factor holds 8 n0^2 bytes (7.2 GB at the bound)
WIDTH = modes.block_width(12)   # columns of every level buffer: the widest LOBPCG block
SINGULAR_PIVOT = 1e-12     # a coarse Cholesky pivot below this times the largest diagonal entry counts as singular


def dof_mask(n_nodes, fixed, dev):
    """uint8 [3 n_nodes] mask, 0 on the three dofs of every fixed node (node ids or a bool node mask)."""
    mask = torch.ones((n_nodes, 3), device=dev, dtype=torch.uint8)
    f = torch.as_tensor(fixed).to(dev) if fixed is not None else None
    if f is not None and f.numel():
        mask[f if f.dtype == torch.bool else f.long()] = 0
    return mask.reshape(-1).contiguous()


class Level:
    """One mesh of the hierarchy: A_s, mask, dinv, the transfers to the next coarser level (None on level 0), buffers."""

    def __init__(self, coords, tets, fixed_fn, E, nu, rho, shift, dev, element_module, parents=None, keep_km=False):
        self.nodes, self.tets = coords.shape[0], tets.shape[0]
        self.n = 3 * self.nodes
        plan = self.plan = ops.CsrPlan(tets, self.nodes, dev)
        brow, bcol = plan.pattern(1)
        keep_m = keep_km and rho is not None   # rho None: K alone (buckling needs no mass)
        Ke = element_module.compute_c3d4_K_matrix(coords, tets, E, nu, device=dev, dtype=torch.float64)
        Me = element_module.compute_c3d4_M_matrix(coords, tets, rho, device=dev, dtype=torch.float64) if (shift or keep_m) else None
        self.K = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ke, 3)) if (keep_km or not shift) else None
        self.M = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Me, 3)) if keep_m else None
        self.A = self.K if not shift else ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ke + shift * Me, 3))
        del Ke, Me
        self.mask = dof_mask(self.nodes, fixed_fn(coords), dev)
        self.dinv = self.A.jacobi(self.mask)
        self.P = self.R = None
        if parents is not None:
            nc = self.nodes - parents.shape[0]
            self.P = hybrid._prolongation_csr(parents, nc, dev)
            self.R = hybrid._restriction_csr(parents, nc, dev)
        self.b, self.x, self.y, self.t = (level_buffer(self.n, dev) for _ in range(4))

    def restrict(self, coarse, na, X, stream):
        """coarse.b[:, :na] = coarse.mask (R X) (femb_mg_transfer)."""
        _node_transfer(self.R, coarse.nodes, self.nodes, coarse.mask, na, X, coarse.b, False, stream)

    def prolong(self, coarse, na, Xc, Y, stream):
        """Y[:, :na] += mask (P Xc) (femb_mg_transfer)."""
        _node_transfer(self.P, self.nodes, coarse.nodes, self.mask, na, Xc, Y, True, stream)


def level_buffer(n, dev):
    return torch.zeros((n, WIDTH), device=dev, dtype=torch.float64)


def _node_transfer(S, n_out, n_in, mask_out, na, X, Y, accumulate, stream):
    crow, col, val = S
    with torch.cuda.device(X.device):
        check(lib.femb_mg_transfer(n_out, n_in, col.numel(), _p(crow), _p(col), _p(val), _p(mask_out), na, _p(X), WIDTH, int(accumulate),
                                   _p(Y), WIDTH, stream), "femb_mg_transfer")


def dense_free_block(A, mask):
    """(free dof ids, dense A[free][:, free]) of a 3x3 block-CSR operator."""
    rows = torch.repeat_interleave(torch.arange(A.nb, device=A.dev), (A.brow[1:] - A.brow[:-1]).long())
    D = torch.zeros((3 * A.nb, 3 * A.nb), device=A.dev, dtype=torch.float64)
    d = torch.arange(3, device=A.dev)
    D[(3 * rows[:, None, None] + d[:, None]), (3 * A.bcol.long()[:, None, None] + d[None, :])] = A.bval
    idx = torch.nonzero(mask).reshape(-1)
    return idx, D[idx][:, idx]


class Hierarchy:
    """V-cycle over levels L[0] (coarsest, dense Cholesky) .. L[-1] (finest).  A level holds A (ops.Bsr3), mask, dinv, nodes, n, the
    buffers b, x, y, t and, above level 0, restrict / prolong to the level below (femb200/amg.py builds such levels algebraically).
    Here they come from a coarse C3D4 mesh (coords, tets) + `levels` uniform refinements; `fixed_fn(coords_l)` gives the clamped
    node ids of every level.  `self.L[-1]` is the finest level; its K and M (shift-free) are kept for LOBPCG
    (rho = None with shift = 0: no mass is assembled, the finest level keeps K only)."""

    def __init__(self, coords, tets, levels, fixed_fn, E, nu, rho, shift, dev, element_module):
        self.dev, self.shift = dev, float(shift)
        coords = torch.as_tensor(coords).to(dev, torch.float64)
        tets = torch.as_tensor(tets).to(dev).long()
        mesh = [(coords, tets, None)]
        for _ in range(levels):
            coords, tets, parents = hybrid.refine_once(coords, tets, element_module)
            mesh.append((coords, tets, parents))
        self.coords, self.tets = coords, tets
        # level 0 first: its dense factor is the one step that can refuse the problem
        self.L = [Level(*mesh[0][:2], fixed_fn, E, nu, rho, shift, dev, element_module, keep_km=levels == 0)]
        self._factor(self.L[0])
        for k, (c, t, parents) in enumerate(mesh[1:], 1):
            self.L.append(Level(c, t, fixed_fn, E, nu, rho, shift, dev, element_module, parents, keep_km=k == levels))
        self.stream = torch.cuda.current_stream(dev).cuda_stream

    def _factor(self, l0):
        nf = int(l0.mask.sum())
        if nf > MAX_COARSE_DOFS:
            raise ValueError(f"the coarse mesh has {nf} free dofs; its dense factor allows at most {MAX_COARSE_DOFS}: refine a coarser mesh more often")
        idx, A0 = dense_free_block(l0.A, l0.mask)
        L, info = torch.linalg.cholesky_ex(A0)
        d = torch.diagonal(L)
        if int(info) != 0 or nf and float((d * d).min()) < SINGULAR_PIVOT * float(torch.diagonal(A0).max()):
            raise ValueError("the coarse operator K + shift M is singular on the free dofs (a free-free or under-constrained model): "
                             "pass shift > 0")
        self.idx0, self.chol0 = idx, L
        self.g0 = torch.zeros((nf, WIDTH), device=self.dev, dtype=torch.float64)

    def describe(self):
        return [{"nodes": lv.nodes, "tets": lv.tets, "dofs": lv.n} for lv in self.L]

    # ---------------------------------------------------------------------------------------------- kernels
    def smooth(self, lv, na, X_in, X_out, out_c0=0, res=None):
        """One damped-Jacobi step on lv.b (columns :na): X_out[:, c0:] = X_in + OMEGA dinv (b - A X_in), X_in None = 0; res = b - A X_in."""
        A = lv.A
        with torch.cuda.device(self.dev):
            check(lib.femb_mg_smooth_bsr3(A.nb, A.nnzb, _p(A.brow), _p(A.bcol), _p(A.bval), _p(lv.mask), _p(lv.dinv), OMEGA, na,
                                          _p(lv.b), WIDTH, _p(X_in), WIDTH, _p(X_out, out_c0), X_out.shape[1] if X_out is not None else 0,
                                          _p(res), WIDTH, self.stream), "femb_mg_smooth_bsr3")

    def coarse_solve(self):
        """L[0].x = A_0^-1 L[0].b on the free dofs (all WIDTH columns: a fixed shape keeps the library's path, and the result, fixed)."""
        l0 = self.L[0]
        torch.index_select(l0.b, 0, self.idx0, out=self.g0)
        l0.x.index_copy_(0, self.idx0, torch.cholesky_solve(self.g0, self.chol0))
        return l0.x

    def cycle(self, l, na, out=None, c0=0):
        """V-cycle on level l with right-hand side L[l].b (columns :na).  The result lands in one of the level's buffers (returned),
        or, when `out` is given, the last smoothing step writes it to out[:, c0:c0+na] (any leading dimension)."""
        if l == 0:
            x = self.coarse_solve()
            if out is not None:
                out[:, c0:c0 + na].copy_(x[:, :na])
            return x
        lv, cl = self.L[l], self.L[l - 1]
        x, y = lv.x, lv.y
        self.smooth(lv, na, None, x)
        for _ in range(SMOOTH - 1):
            self.smooth(lv, na, x, y)
            x, y = y, x
        self.smooth(lv, na, x, None, res=lv.t)
        lv.restrict(cl, na, lv.t, self.stream)
        xc = self.cycle(l - 1, na)
        lv.prolong(cl, na, xc, x, self.stream)
        for s in range(SMOOTH):
            if s == SMOOTH - 1 and out is not None:
                self.smooth(lv, na, x, out, c0)
                return out
            self.smooth(lv, na, x, y)
            x, y = y, x
        return x

    def apply(self, B):
        """Preconditioner on a [n_fine, k <= 16] tensor (masked rows in, masked rows out): returns V(B) as a new tensor."""
        top = self.L[-1]
        k = B.shape[1]
        top.b[:, :k].copy_(B)
        out = torch.empty((top.n, k), device=self.dev, dtype=torch.float64)
        self.cycle(len(self.L) - 1, k, out, 0)
        return out


class MultilevelBackend(modes.DeviceBackend):
    """LOBPCG backend whose residual step preconditions with the V-cycle instead of Jacobi.  The pencil (A, B) defaults to the finest
    level's (K, M); mask: the finest level's."""

    def __init__(self, H, A=None, B=None):
        top = H.L[-1]
        super().__init__(top.K if A is None else A, top.M if B is None else B, top.mask)
        self.H = H
        self.maskf = top.mask.to(torch.float64)

    def residual(self, X, KX, MX, m, lam, active, na, W, c0, norms):
        """As DeviceBackend.residual, but W[:, c0+a] = V(r_active[a]): the masked residuals go to the finest level's rhs buffer
        (the float mask as dinv), the cycle's last smoothing step writes W."""
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        top = self.H.L[-1]
        with torch.cuda.device(self.dev):
            check(lib.femb_lobpcg_residual(X.shape[0], m, _p(X), X.shape[1], _p(KX), _p(MX), KX.shape[1], lam.ctypes.data_as(C.POINTER(C.c_double)),
                                           _p(self.maskf), na, _p(active), _p(top.b), WIDTH, _p(norms), self.stream), "femb_lobpcg_residual")
        if na:
            self.H.cycle(len(self.H.L) - 1, na, W, c0)
