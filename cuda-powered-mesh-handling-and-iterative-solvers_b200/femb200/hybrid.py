"""Hybrid subdivided-mesh solver: direct solve on a coarse mesh + iterative CG on its uniform refinements
(BASELINE config 5, "direct coarse solve + iterative CG on 3-level refined tet mesh").

What the reference has (SURVEY.md section 3E): `README.md:7` names a "hybrid solver of iterative and inverse methods with
sub-divided mesh"; `subdivision.ipynb` builds per-subdomain dense inverses and stops before any solve loop.  The pieces that
DO exist and that this module composes are: one uniform 8-way refinement = `c3d4_to_c3d10` (mid-edge insertion,
element.py:777-833) followed by `c3d10_to_c3d4` (element.py:963-993); the `u_init` warm start of every CG solver
(solver.py:166-169); and the CG loop itself (solver.py:144-229, pinned).  The coarse direct solve and the prolongation have
no counterpart in the reference -- parity unpinned -- and are validated against a single-level CG solve of the same fine
problem (tests/test_gpu_parity.py::test_hybrid_cascade).

Two modes.  `mode="multilevel"` (default): the direct coarse solve and the refined levels work TOGETHER inside the iteration --
CG on the finest level preconditioned by one symmetric V-cycle over the mesh hierarchy (damped-Jacobi smoothing on the refined
levels, restriction = transpose of the prolongation below, dense Cholesky solve on level 0).  On BASELINE config 5 (n=8 coarse
cube, 3 refinements, 824 k dofs) this converges in ~20 iterations where CG on the fine mesh alone needs ~1300.
`mode="cascade"`: the round-1 scheme, kept for comparison -- it saved 7 % of the iterations and cost wall time.

Cascade: level 0 is solved directly (dense Cholesky of the constrained operator: a cuSOLVER library call, which SURVEY 2.2
allows for the coarse solve); the solution is prolongated to the next level (a mid-edge node receives the mean of its two
parents, which is exactly how element.py:814 places the node, so P1 functions are reproduced exactly) and used as `u_init`
of the reference CG loop on that level's assembled operator; repeat up to the finest level.
"""
from __future__ import annotations

import os

import torch

from . import ops


def refine_once(coords, tets, element_module):
    """One uniform refinement with the reference's own building blocks.  Returns (coords', tets', parents [N'-N, 2])."""
    dev = coords.device
    N = coords.shape[0]
    c10, e10, _, _ = element_module.c3d4_to_c3d10(coords, tets, dtype=coords.dtype, device=dev)
    e10 = e10.long()
    # parents of every inserted node, from the element table: slot 4..9 <-> edges (0,1),(1,2),(2,0),(0,3),(1,3),(2,3)
    slots = torch.tensor([[0, 1], [1, 2], [2, 0], [0, 3], [1, 3], [2, 3]], device=dev)
    mids = e10[:, 4:].reshape(-1) - N
    pa = e10[:, slots].reshape(-1, 2)
    parents = torch.empty((c10.shape[0] - N, 2), dtype=torch.int64, device=dev)
    parents[mids] = pa
    return c10, element_module.c3d10_to_c3d4(e10, device=dev), parents


def prolongate(u, parents):
    """Linear interpolation to the refined mesh: old nodes keep their value, a mid-edge node takes the parents' mean."""
    return torch.cat([u, 0.5 * (u[parents[:, 0]] + u[parents[:, 1]])], dim=0)


def _restriction_csr(parents, n_coarse, dev):
    """R = P^T as CSR [n_coarse, n_coarse + n_mid]: 1 on the node itself, 1/2 on every mid-edge child (applied with the
    library's deterministic SpMV; an index_add_ scatter would sum in atomic order)."""
    nm = parents.shape[0]
    rows = torch.cat([torch.arange(n_coarse, device=dev), parents[:, 0], parents[:, 1]])
    cols = torch.cat([torch.arange(n_coarse, device=dev), n_coarse + torch.arange(nm, device=dev), n_coarse + torch.arange(nm, device=dev)])
    vals = torch.cat([torch.ones(n_coarse, device=dev, dtype=torch.float64), torch.full((2 * nm,), 0.5, device=dev, dtype=torch.float64)])
    key = torch.sort(rows * (n_coarse + nm) + cols).indices
    rows, cols, vals = rows[key], cols[key], vals[key]
    crow = torch.zeros(n_coarse + 1, dtype=torch.int64, device=dev)
    crow[1:] = torch.cumsum(torch.bincount(rows, minlength=n_coarse), 0)
    return crow.to(torch.int32).contiguous(), cols.to(torch.int32).contiguous(), vals.contiguous()


def _prolongation_csr(parents, n_coarse, dev):
    """P as CSR [n_coarse + n_mid, n_coarse], the matrix of `prolongate`: row i < n_coarse holds (i, 1), row n_coarse + k holds
    (parents[k], 1/2) with the two columns ascending."""
    nm = parents.shape[0]
    pc = torch.sort(parents, dim=1).values
    cols = torch.cat([torch.arange(n_coarse, device=dev), pc.reshape(-1)])
    vals = torch.cat([torch.ones(n_coarse, device=dev, dtype=torch.float64), torch.full((2 * nm,), 0.5, device=dev, dtype=torch.float64)])
    crow = torch.cat([torch.arange(n_coarse + 1, device=dev), n_coarse + 2 * torch.arange(1, nm + 1, device=dev)])
    return crow.to(torch.int32).contiguous(), cols.to(torch.int32).contiguous(), vals.contiguous()


def multilevel_solve(coords, tets, levels, load_fn, fixed_fn, E=None, nu=None, kind="elasticity", tol=1e-8, max_iter=500, device="cuda:0",
                     element_module=None, verbose=False, smooth=2, omega=0.6):
    """CG on the finest mesh preconditioned by a V(smooth, smooth) cycle over the hierarchy coarse mesh + `levels` uniform
    refinements; level 0 is solved directly (dense Cholesky).  Convergence test as the reference's CG: sqrt(r.r) < tol on the
    projected residual (solver.py:208-212).  Returns (u_fine, coords_fine, tets_fine, info)."""
    if element_module is None:
        import element as element_module
    dev = ops.cuda_device(device)
    coords = torch.as_tensor(coords).to(dev, torch.float64)
    tets = torch.as_tensor(tets).to(dev).long()
    ndof = 3 if kind == "elasticity" else 1
    L = []          # per level: dict(apply, dinv, free [N,ndof] float mask, parents, R)

    def build_level(c, t, parents):
        plan = ops.CsrPlan(t, c.shape[0], dev)
        vals = plan.assemble_c3d4(c, kind, E or 0.0, nu or 0.0)
        free = torch.ones((c.shape[0], ndof), dtype=torch.float64, device=dev)
        free[fixed_fn(c).to(dev).long()] = 0.0
        if ndof == 3:
            brow, bcol = plan.pattern(1)
            A = ops.Bsr3.from_csr_values(brow, bcol, vals)
            apply = lambda x: A.spmv(x * free) * free  # noqa: E731  (projected operator: fixed dofs stay zero)
            dinv = A.jacobi().reshape(-1, 3) * free             # 1 / diag (0 where the diagonal vanishes)
        else:
            crow, col = plan.pattern(1)
            apply = lambda x: ops.spmv(crow, col, vals, x * free) * free  # noqa: E731
            dinv = ops.jacobi(crow, col, vals).reshape(-1, 1) * free
        lev = {"apply": apply, "dinv": dinv, "free": free, "parents": parents, "plan": plan, "vals": vals, "nodes": c.shape[0], "tets": t.shape[0]}
        if parents is not None:
            lev["R"] = _restriction_csr(parents, c.shape[0] - parents.shape[0], dev)
        return lev

    L.append(build_level(coords, tets, None))
    for _ in range(levels):
        coords, tets, parents = refine_once(coords, tets, element_module)
        L.append(build_level(coords, tets, parents))
    # level 0: dense Cholesky of the constrained operator
    l0 = L[0]
    n0 = l0["nodes"] * ndof
    crow0, col0 = l0["plan"].pattern(ndof)
    A0 = torch.sparse_csr_tensor(crow0, col0, l0["vals"], size=(n0, n0)).to_dense()
    idx0 = torch.nonzero(l0["free"].reshape(-1) > 0).reshape(-1)
    chol0 = torch.linalg.cholesky(A0[idx0][:, idx0])
    del A0

    def coarse_solve(r):
        x = torch.zeros(n0, dtype=torch.float64, device=dev)
        x[idx0] = torch.cholesky_solve(r.reshape(-1)[idx0].unsqueeze(1), chol0).squeeze(1)
        return x.reshape(-1, ndof)

    def restrict(lev, r):
        crow, col, val = lev["R"]
        return torch.stack([ops.spmv(crow, col, val, r[:, k].contiguous()) for k in range(ndof)], dim=1)

    def vcycle(l, r):
        if l == 0:
            return coarse_solve(r)
        lev = L[l]
        x = omega * lev["dinv"] * r
        for _ in range(smooth - 1):
            x = x + omega * lev["dinv"] * (r - lev["apply"](x))
        rc = restrict(lev, r - lev["apply"](x)) * L[l - 1]["free"]
        x = x + prolongate(vcycle(l - 1, rc), lev["parents"]) * lev["free"]
        for _ in range(smooth):
            x = x + omega * lev["dinv"] * (r - lev["apply"](x))
        return x

    top = L[-1]
    F = load_fn(coords, tets).to(dev, torch.float64).reshape(-1, ndof) * top["free"]
    u = torch.zeros_like(F)
    r = F.clone()
    z = vcycle(levels, r)
    p = z.clone()
    rz = float((r * z).sum())
    its, status = 0, "maxiter"
    for i in range(max_iter):
        Ap = top["apply"](p)
        alpha = rz / float((p * Ap).sum())
        u += alpha * p
        r -= alpha * Ap
        its = i + 1
        rs = float((r * r).sum())
        if rs ** 0.5 < tol:
            status = "converged"
            break
        z = vcycle(levels, r)
        rz_new = float((r * z).sum())
        p = z + (rz_new / rz) * p
        rz = rz_new
    info = {"kind": kind, "mode": "multilevel", "iterations": its, "status": status, "rs": rs if its else 0.0,
            "levels": [{"nodes": lv["nodes"], "tets": lv["tets"], "solver": "dense Cholesky" if k == 0 else f"V({smooth},{smooth}) damped Jacobi"}
                       for k, lv in enumerate(L)]}
    info["levels"][-1].update(iterations=its, status=status)
    if verbose:
        print(f"multilevel PCG: {its} iterations ({status}), {top['nodes']} nodes / {top['tets']} tets on the finest of {levels + 1} levels")
    return u, coords, tets, info


def hybrid_solve(coords, tets, levels, load_fn, fixed_fn, E=None, nu=None, kind="elasticity", tol=1e-8, max_iter=10000, device="cuda:0",
                 element_module=None, verbose=False, mode="multilevel"):
    """coords/tets: coarse C3D4 mesh.  load_fn(coords_l, tets_l) -> F [N_l, ndof]; fixed_fn(coords_l) -> fixed node ids.
    kind: 'elasticity' (3 dofs, E/nu) or 'poisson' (1 dof).  Returns (u_fine, coords_fine, tets_fine, info).
    mode: 'multilevel' (V-cycle preconditioned CG, see the module docstring) or 'cascade' (prolongation-only warm starts)."""
    if mode == "multilevel" and levels >= 1:
        return multilevel_solve(coords, tets, levels, load_fn, fixed_fn, E, nu, kind, tol, min(max_iter, 2000), device, element_module, verbose)
    if element_module is None:
        import element as element_module  # the drop-in mirror (solver/ is on sys.path when used through solver.py)
    dev = ops.cuda_device(device)
    coords = torch.as_tensor(coords).to(dev, torch.float64)
    tets = torch.as_tensor(tets).to(dev).long()
    ndof = 3 if kind == "elasticity" else 1
    info = {"levels": [], "kind": kind}

    plans = {}

    def operator(c, t):
        plan = plans[t.data_ptr()] = ops.CsrPlan(t, c.shape[0], dev)
        crow, col = plan.pattern(ndof)
        vals = plan.assemble_c3d4(c, kind, E or 0.0, nu or 0.0)
        return crow, col, vals

    def bsr_of(c, t, vals):
        brow, bcol = plans[t.data_ptr()].pattern(1)
        return ops.Bsr3.from_csr_values(brow, bcol, vals)

    # ---- level 0: direct solve of the constrained system (fixed dofs replaced by identity rows/columns)
    crow, col, vals = operator(coords, tets)
    n = coords.shape[0] * ndof
    A = torch.sparse_csr_tensor(crow, col, vals, size=(n, n)).to_dense()
    F = load_fn(coords, tets).to(dev, torch.float64).reshape(-1)
    free = torch.ones((coords.shape[0], ndof), dtype=torch.bool, device=dev)
    free[fixed_fn(coords).to(dev).long()] = False
    free = free.reshape(-1)
    idx = torch.nonzero(free).reshape(-1)
    L = torch.linalg.cholesky(A[idx][:, idx])
    u = torch.zeros(n, dtype=torch.float64, device=dev)
    u[idx] = torch.cholesky_solve(F[idx].unsqueeze(1), L).squeeze(1)
    u = u.reshape(-1, ndof)
    info["levels"].append({"nodes": coords.shape[0], "tets": tets.shape[0], "solver": "dense Cholesky", "iterations": 0})
    # ---- refined levels: prolongate, warm-started CG
    for lvl in range(1, levels + 1):
        coords, tets, parents = refine_once(coords, tets, element_module)
        u0 = prolongate(u, parents)
        crow, col, vals = operator(coords, tets)
        F = load_fn(coords, tets).to(dev, torch.float64)
        mask = torch.ones((coords.shape[0], ndof), dtype=torch.uint8, device=dev)
        mask[fixed_fn(coords).to(dev).long()] = 0
        kw = dict(mask=mask.reshape(-1).contiguous(), u_init=u0, tol=tol, max_iter=max_iter)
        if ndof == 3 and not os.environ.get("FEMB_NO_BSR"):   # elasticity: 3x3 block-CSR inner CG
            u, it = bsr_of(coords, tets, vals).cg_solve(F.reshape(-1, ndof), **kw)
        else:
            u, it = ops.cg_solve(crow, col, vals, F.reshape(-1, ndof), **kw)
        u = u.reshape(-1, ndof)
        info["levels"].append({"nodes": coords.shape[0], "tets": tets.shape[0], "solver": "CG (warm start from the coarser level)",
                               "iterations": it["iterations"], "status": it["status"]})
        if verbose:
            print(f"level {lvl}: {coords.shape[0]} nodes, {tets.shape[0]} tets, CG {it['iterations']} iterations ({it['status']})")
    return u, coords, tets, info
