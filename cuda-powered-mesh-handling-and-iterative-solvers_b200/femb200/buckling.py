"""Linear (eigenvalue) buckling of solid meshes: the load multipliers at which the stiffness of a prestressed part vanishes.

With u_ref = K^-1 F the linear static response to the reference load F and K_G = K_G(u_ref) the geometric stiffness of its stress
(femb_solid_geometric), the critical states satisfy (K + lam K_G) phi = 0.  The solver works on the symmetric-definite pencil

    K_G phi = nu K phi        on the free dofs,   lam = -1 / nu  for nu < 0,   lam = +inf for nu >= 0 (no buckling in that pair),

so the lowest nu give the lowest load factors in ascending order, and LOBPCG (femb200/modes.py) runs on it unchanged with A = K_G and
B = K: K_G and K are assembled on one plan, so femb_spmm_bsr3 reads both blocks of a nonzero in one pass.  The ideal preconditioner
of the pencil is K^-1, the inverse of B; both backends precondition with B:
  - `JacobiBackend`: diag(K)^-1 (not diag(K_G)^-1, which is indefinite and can be zero);
  - `MultilevelBackend`: one V-cycle of femb200/multigrid.py at shift 0, K_G on the finest level only.
The modes come out K-orthonormal with zeros on the fixed dofs.  An unconverged reference solve raises a ValueError: the load factors
of an inexact prestress would be wrong without any sign of it.
"""
from __future__ import annotations

import numpy as np
import torch

from . import modes, multigrid


class JacobiBackend(modes.DeviceBackend):
    """LOBPCG backend of the pencil (K_G, K) with the Jacobi preconditioner of B = K."""

    def __init__(self, KG, K, mask):
        super().__init__(KG, K, mask)
        self.dinv = K.jacobi(mask)


class MultilevelBackend(multigrid.MultilevelBackend):
    """LOBPCG backend of the pencil (K_G, K) preconditioned by the V-cycle of H (shift 0), K = the finest level's K."""

    def __init__(self, H, KG):
        super().__init__(H, KG, H.L[-1].K)


def load_factors(nu):
    """lam_i = -1 / nu_i for nu_i < 0, +inf otherwise (ascending when nu is)."""
    nu = np.asarray(nu, dtype=np.float64)
    with np.errstate(divide="ignore"):
        return np.where(nu < 0.0, -1.0 / np.where(nu < 0.0, nu, -1.0), np.inf)


def _rhs(F, mask):
    """The load on the free dofs as one fp64 vector, and its norm; a zero load is refused."""
    maskf = mask.to(torch.float64)
    b = torch.as_tensor(F).to(mask.device, torch.float64).reshape(-1) * maskf
    if b.numel() != mask.numel():
        raise ValueError(f"the load must be [N, 3] with N = {mask.numel() // 3}, got {b.numel()} values")
    bn = float(torch.linalg.vector_norm(b))
    if not bn > 0.0:
        raise ValueError("the reference load is zero on the free dofs: buckling needs a nonzero load")
    return b, bn, maskf


def _refuse(kind, res, its, tol):
    raise ValueError(f"the reference static solve ({kind}) did not converge: relative residual |F - K u| / |F| = {res:.3e} after {its} "
                     f"iterations, static_tol = {tol:.1e} (an unconstrained or under-constrained model, or raise static_max_iter)")


def static_jacobi(K, mask, F, tol, max_iter):
    """u_ref = K^-1 F on the free dofs with the device Jacobi-PCG (Bsr3.cg_solve).  That loop stops on sqrt(r . D^-1 r); the threshold
    tol |F| sqrt(min D^-1) makes it imply |r| <= tol |F|.  Returns (u [3N], iterations, |F - K u| / |F|)."""
    b, bn, maskf = _rhs(F, mask)
    minv = K.jacobi(mask)
    dmin = float(minv[mask != 0].min())
    u, info = K.cg_solve(b, mask=mask, minv=minv, tol=tol * bn * np.sqrt(max(dmin, 0.0)), max_iter=max_iter, eps=0.0)
    res = float(torch.linalg.vector_norm((b - K.spmv(u)) * maskf)) / bn
    if info["status"] != "converged" or not np.isfinite(res):
        _refuse("Jacobi-PCG", res, info["iterations"], tol)
    return u, info["iterations"], res


def static_multigrid(H, F, tol, max_iter):
    """u_ref = K^-1 F on the finest level of H by PCG with one V-cycle (Hierarchy.apply) per iteration, stopped at |r| <= tol |F|
    (host scalars per iteration: a few tens of iterations).  Returns (u [3N], iterations, |F - K u| / |F|)."""
    top = H.L[-1]
    K = top.K
    b, bn, maskf = _rhs(F, top.mask)
    x = torch.zeros_like(b)
    r = b.clone()
    z = H.apply(r[:, None])[:, 0]
    p = z.clone()
    rz = float(torch.dot(r, z))
    rn, it = bn, 0
    while rn > tol * bn and it < max_iter:
        q = K.spmv(p) * maskf
        alpha = rz / float(torch.dot(p, q))
        x.add_(p, alpha=alpha)
        r.add_(q, alpha=-alpha)
        rn = float(torch.linalg.vector_norm(r))
        it += 1
        if not np.isfinite(rn) or rn <= tol * bn:
            break
        z = H.apply(r[:, None])[:, 0]
        rz_new = float(torch.dot(r, z))
        p.mul_(rz_new / rz).add_(z)
        rz = rz_new
    res = float(torch.linalg.vector_norm((b - K.spmv(x)) * maskf)) / bn
    if not rn <= tol * bn or not np.isfinite(res):
        _refuse("multigrid PCG", res, it, tol)
    return x, it, res


def solve(be, num_eigs, tol, max_iter):
    """LOBPCG on the pencil held by `be`.  Returns (load factors [num_eigs] ascending, modes [n, num_eigs] (K-orthonormal, in the
    backend's memory), info: the LOBPCG fields without freq_hz, plus nu)."""
    nu, S, info = modes.lobpcg(be, num_eigs, tol=tol, max_iter=max_iter)
    del info["freq_hz"]
    info["nu"] = nu.copy()
    return load_factors(nu), _k_orthonormalise(be, S, num_eigs), info


def _k_orthonormalise(be, S, k):
    """X = S[:, :k] L^-T with L L^T = X^T (K X) from a fresh SpMM.  LOBPCG carries K S by recurrence (combines of earlier products);
    with B = K, whose condition number grows like h^-2 and with slenderness, that Gram drifts from I by about eps cond(K) (3e-9 on a
    1 x 1 x 20 C3D4 column, 6e-12 after this step)."""
    YA, YB = be.zeros(be.n, k), be.zeros(be.n, k)
    be.spmm(S, 0, k, YA, YB)
    g = be.zeros(1, k * k).reshape(-1)
    be.gram(S, YB, k, g)
    G = be.host(g).reshape(k, k)
    L = np.linalg.cholesky(0.5 * (G + G.T))
    X = be.zeros(be.n, k)
    be.combine(S, k, np.linalg.inv(L).T, X, 0)
    return X
