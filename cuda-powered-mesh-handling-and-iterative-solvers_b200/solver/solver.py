"""Drop-in mirror of the CG family of the reference's `solver/solver.py` on sm_100a kernels.

Same names, argument order, defaults and return values as the reference.  Where the reference applies the
operator element by element in every iteration (gather -> bmm -> atomic index_add, solver.py:184), these solvers
assemble the operator once into CSR (deterministic sort-based assembly) and run the whole loop on the device:
three fused kernels per iteration captured in a CUDA graph, scalars never leave the GPU, and the convergence /
breakdown tests are the reference's own (absolute sqrt(r.r) < tol, +eps denominators, pAp guards, node-level
fixing by projection).  Each solver also accepts `return_info=True` (additive) to get the iteration count the
reference only prints.
"""
from __future__ import annotations

import os
import sys

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
if _HERE not in sys.path:
    sys.path.insert(0, _HERE)

from element import *  # noqa: E402,F401,F403  (the reference does the same: solver.py:1-2)
from shell import *    # noqa: E402,F401,F403
import element as _el  # noqa: E402
import shell as _sh    # noqa: E402
from femb200 import ops as _ops  # noqa: E402


def _dof_mask(n_nodes, ndof, fixed, dev):
    mask = torch.ones((n_nodes, ndof), device=dev, dtype=torch.uint8)
    if fixed is not None and torch.as_tensor(fixed).numel():
        f = torch.as_tensor(fixed).to(dev)
        # u[rbe2] = 0 in the reference (solver.py:161) accepts an index list or a boolean node mask
        mask[f if f.dtype == torch.bool else f.long()] = 0
    return mask.reshape(-1).contiguous()


def _report(kind, info, max_iter):
    # the reference prints these lines (solver.py:188-226); kept so notebook output reads the same
    if info["status"] == "converged":
        print(f"Converged after {info['iterations']} iterations. Residual norm: {info['rs']:.3e}")
    elif info["status"] == "breakdown":
        print(f"Terminating early at iteration {info['iterations']}: CG breakdown (p^T K p invalid or NaN/Inf step).")
    else:
        print(f"{kind} did not converge within the maximum number of iterations.")


def _operator(K, elements, N, dev):
    """CSR of sum_e K_e (or pass-through of an already assembled torch CSR tensor)."""
    if isinstance(K, torch.Tensor) and K.layout == torch.sparse_csr:
        return K.crow_indices().to(torch.int32), K.col_indices().to(torch.int32), K.values().to(torch.float64), None
    K = torch.as_tensor(K)
    ndof = K.shape[1] // elements.shape[1]
    plan = _ops.cached_plan(elements, N, dev)
    crow, col = plan.pattern(ndof)
    return crow, col, plan.assemble(K, ndof), plan


class _Assembled:
    """The assembled operator of one solve.  3-dof operators (every elasticity operator of the reference,
    dofs = node*3+{0,1,2}) are stored as 3x3 block-CSR: 8.44 instead of 12 bytes per nonzero and a third of the x gathers
    per SpMV; everything else (and FEMB_NO_BSR=1, for A/B runs) takes scalar CSR."""

    def __init__(self, K, elements, N, ndof, dev):
        crow, col, val, plan = _operator(K, elements, N, dev)
        self.bsr = None
        if plan is not None and ndof == 3 and not os.environ.get("FEMB_NO_BSR"):
            brow, bcol = plan.pattern(1)
            self.bsr = _ops.Bsr3.from_csr_values(brow, bcol, val)
        else:
            self.csr = (crow, col, val)

    def spmv(self, x):
        return self.bsr.spmv(x) if self.bsr is not None else _ops.spmv(*self.csr, x)

    def cg_solve(self, F, **kw):
        return self.bsr.cg_solve(F, **kw) if self.bsr is not None else _ops.cg_solve(*self.csr, F, **kw)


def _cg(K, elements, F, dev, **kw):
    """Assemble once and run the device loop."""
    N, ndof = F.shape
    return _Assembled(K, elements, N, ndof, dev).cg_solve(F, **kw)


def _distributed_world():
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def stable_conjugate_gradient_solver(K, elements, F, rbe2, u_init=None, tol=1e-10, max_iter=1000, device="cuda:0", dtype=torch.float64,
                                     eps=1e-30, return_info=False, verbose=True, distributed=False, coords=None):
    """Projected CG with node fixing (solver.py:144-229).  K: element matrices [M,nd,nd] (assembled internally) or a
    torch CSR tensor.  Arithmetic is fp64 (the reference's default); the result is cast to `dtype`.
    `distributed=True` (additive; one process per GPU with torch.distributed initialised, every rank passing the same
    arguments): rows are partitioned over the ranks -- by recursive coordinate bisection when `coords` is given, by node-id
    ranges otherwise -- each rank assembles its rows from K and the loop runs over NVLink peer memory (femb200.dist_cg); the
    full solution is returned on every rank.  Same iterates as the single-GPU loop up to summation order."""
    dev = _ops.cuda_device(device)
    F = torch.as_tensor(F).to(dev)
    N, ndof = F.shape
    if distributed and _distributed_world() > 1:
        from femb200 import dist_cg
        if K.layout == torch.sparse_csr:
            raise ValueError("distributed=True assembles each rank's rows from element matrices: pass K as [M,nd,nd]")
        u, info = dist_cg.solve_replicated(K, elements, F, rbe2, u_init=u_init, tol=tol, max_iter=max_iter, eps=eps, coords=coords, device=dev)
    else:
        u, info = _cg(K, elements, F, dev, mask=_dof_mask(N, ndof, rbe2, dev), u_init=u_init, tol=tol, max_iter=max_iter, eps=eps)
    if verbose:
        _report("CG", info, max_iter)
    u = u.to(dtype)
    return (u, info) if return_info else u


def final_solver(K, elements, F, rbe2, u_init=None, tol=1e-10, max_iter=1000, device="cuda:0", dtype=torch.float64, eps=1e-30,
                 return_info=False, verbose=True):
    """Same mathematics as stable_conjugate_gradient_solver written out of place with a 0/1 mask in the reference
    (solver.py:231-295); identical iterates, so it shares the device loop."""
    return stable_conjugate_gradient_solver(K, elements, F, rbe2, u_init, tol, max_iter, device, dtype, eps, return_info, verbose)


def _shell_global_K(K, unit):
    """T^T K T with T = blockdiag(R,R,...) per node: the element operator of shell.py:58-102 in global axes (one kernel)."""
    return _ops.shell_rotate_K(K, unit)


def stable_conjugate_gradient_shell_solver(K, elements, F, rbe2, coords=None, unit=None, u_init=None, tol=1e-10, max_iter=1000,
                                           device="cuda:0", dtype=torch.float64, eps=1e-30, return_info=False, verbose=True):
    """Shell CG on 6 dofs per node (solver.py:297-389).  The element operator R^T K_e R is assembled once."""
    dev = _ops.cuda_device(device)
    F = torch.as_tensor(F).to(dev)
    if unit is None:
        if coords is None:
            raise ValueError("Neither coords or units data were provided")
        unit = _sh.compute_s3_local_unitvector(coords, elements, device=dev)
    N = F.shape[0]
    Kg = _shell_global_K(torch.as_tensor(K).to(dev, torch.float64), torch.as_tensor(unit).to(dev, torch.float64))
    crow, col, val, _ = _operator(Kg, elements, N, dev)
    u, info = _ops.cg_solve(crow, col, val, F, mask=_dof_mask(N, 6, rbe2, dev), u_init=u_init, tol=tol, max_iter=max_iter, eps=eps)
    if verbose:
        _report("CG", info, max_iter)
    u = u.to(dtype)
    return (u, info) if return_info else u


# ------------------------------------------------------------------------------------------- SPC / RBE2 / RBE3 constraints

def parse_spc_list(spc_list, device="cuda:0", dtype=torch.float64):
    """[{'node','dofs','value'}] -> (nodes int32 [S], dofs int32 [S], values [S]), one entry per constrained dof
    (solver.py:396-435).  Host loop over the dict list, as in the reference."""
    n, d, v = [], [], []
    for spc in spc_list:
        for dof in spc["dofs"]:
            n.append(spc["node"]); d.append(dof); v.append(spc["value"])
    return (torch.tensor(n, device=device, dtype=torch.int32), torch.tensor(d, device=device, dtype=torch.int32),
            torch.tensor(v, device=device, dtype=dtype))


def parse_rbe2_list(rbe2_list, device="cuda:0"):
    """[{'master','slaves','dofs'}] -> (slaves, masters, dofs) int32 [R] (solver.py:437-476)."""
    s, m, d = [], [], []
    for rb in rbe2_list:
        for slave in rb["slaves"]:
            for dof in rb["dofs"]:
                s.append(slave); m.append(rb["master"]); d.append(dof)
    t = lambda a: torch.tensor(a, device=device, dtype=torch.int32)  # noqa: E731
    return t(s), t(m), t(d)


def parse_rbe3_list(rbe3_list, device="cuda:0", dtype=torch.float64):
    """[{'master','slaves','dofs','weights'}] -> (masters, slaves, dofs, weights, offsets int64 [n+1], weight_sums [n])
    (solver.py:603-651)."""
    m, s, d, w, ws, off = [], [], [], [], [], [0]
    for rb in rbe3_list:
        for i, slave in enumerate(rb["slaves"]):
            for dof in rb["dofs"]:
                m.append(rb["master"]); s.append(slave); d.append(dof); w.append(rb["weights"][i])
        ws.append(sum(rb["weights"]))
        off.append(len(m))
    t = lambda a: torch.tensor(a, device=device, dtype=torch.int32)  # noqa: E731
    return (t(m), t(s), t(d), torch.tensor(w, device=device, dtype=dtype), torch.tensor(off, device=device, dtype=torch.int64),
            torch.tensor(ws, device=device, dtype=dtype))


def apply_loads_to_F(F, load_list):
    """F[node] += force for every {'node','force':[fx,fy,fz]} (solver.py:653-663), in place; one index_put instead of a host
    loop of three element writes per load."""
    if not load_list:
        return
    nodes = torch.tensor([ld["node"] for ld in load_list], device=F.device, dtype=torch.long)
    f = torch.tensor([list(ld["force"]) for ld in load_list], device=F.device, dtype=F.dtype)
    F.index_put_((nodes,), f, accumulate=True)


def enforce_constraints(u, r, spc_nodes, spc_dofs, spc_values, rbe2_slaves, rbe2_masters, rbe2_dofs):
    """RBE2 then SPC, in place (solver.py:478-510)."""
    if rbe2_slaves.numel() > 0:
        s, m, d = rbe2_slaves.long(), rbe2_masters.long(), rbe2_dofs.long()
        u[s, d] = u[m, d]
        r[s, d] = 0.0
    if spc_nodes.numel() > 0:
        n, d = spc_nodes.long(), spc_dofs.long()
        u[n, d] = spc_values.to(u.dtype)
        r[n, d] = 0.0


def new_enforce_constraints(u, r, spc_nodes, spc_dofs, spc_values, rbe2_slaves, rbe2_masters, rbe2_dofs, rbe3_master, rbe3_slaves,
                            rbe3_dofs, rbe3_weights, rbe3_inds, weight_sums):
    """SPC, RBE2, then every RBE3 master dof <- weighted mean of its slaves; r is not touched on RBE3 masters
    (solver.py:665-700).  The reference walks the RBE3 list with `.item()` host syncs per constraint and dof; here the
    weighted sums of all (constraint, dof) pairs are formed by one index_add and written with one index_put."""
    if spc_nodes.numel() > 0:
        n, d = spc_nodes.long(), spc_dofs.long()
        u[n, d] = spc_values.to(u.dtype)
        r[n, d] = 0.0
    if rbe2_slaves.numel() > 0:
        s, m, d = rbe2_slaves.long(), rbe2_masters.long(), rbe2_dofs.long()
        u[s, d] = u[m, d]
        r[s, d] = 0.0
    k = rbe3_inds.numel() - 1
    if k > 0 and rbe3_master.numel() > 0:
        nd = u.shape[1]
        cid = torch.repeat_interleave(torch.arange(k, device=u.device), (rbe3_inds[1:] - rbe3_inds[:-1]).to(u.device))
        key = cid * nd + rbe3_dofs.long()
        sums = torch.zeros(k * nd, device=u.device, dtype=u.dtype).index_add_(0, key, rbe3_weights.to(u.dtype) * u[rbe3_slaves.long(), rbe3_dofs.long()])
        # one RBE3 after the other in the reference: a later master may read an earlier master's fresh value only if it is
        # one of its slaves -- not supported by the vectorised form and rejected here
        uk = torch.unique(key)
        masters = rbe3_master.long()[rbe3_inds[:-1].long().to(u.device)][uk // nd]
        if bool(torch.isin(rbe3_slaves.long(), masters).any()):
            raise ValueError("an RBE3 master is also an RBE3 slave: chained RBE3 constraints are not supported")
        u[masters, uk % nd] = sums[uk] / (weight_sums.to(u.dtype)[uk // nd] + 1e-30)


def _constrained_solve(K, elements, F, spc, rbe2, rbe3, u_init, tol, max_iter, dev, dtype, eps, return_info, verbose):
    """Both constrained CG loops of the reference.  On SPC and RBE2-slave dofs r is zeroed before p = r, so p stays zero there
    and the loop is the dof-masked CG on the remaining dofs; the values written into u on constrained dofs (SPC values,
    RBE2 copies, RBE3 means) never feed back into r.  The device loop therefore solves the masked problem for the
    increment u - u_init and the constraints are written once, in the reference's order, on the final iterate."""
    F = torch.as_tensor(F).to(dev, torch.float64)
    N, nd = F.shape
    A = _Assembled(K, elements, N, nd, dev)
    mask = torch.ones((N, nd), device=dev, dtype=torch.uint8)
    if spc[0].numel():
        mask[spc[0].long(), spc[1].long()] = 0
    if rbe2[0].numel():
        mask[rbe2[0].long(), rbe2[2].long()] = 0
    if u_init is None:
        u0, rhs = torch.zeros_like(F), F
    else:
        u0 = torch.as_tensor(u_init).to(dev, torch.float64).clone()
        rhs = F - A.spmv(u0.reshape(-1)).reshape(N, nd)
    du, info = A.cg_solve(rhs, mask=mask.reshape(-1).contiguous(), tol=tol, max_iter=max_iter, eps=eps)
    u = u0 + du
    scratch = torch.zeros_like(u)
    for _ in range(2):  # the reference enforces after every update: a second pass lets values set late in a pass (an SPC value on
        # an RBE2 master, an RBE2 copy feeding an RBE3 mean) reach their dependants exactly as they do there
        if rbe3 is None:
            enforce_constraints(u, scratch, *spc, *rbe2)
        else:
            new_enforce_constraints(u, scratch, *spc, *rbe2, *rbe3)
    if verbose:
        if info["status"] == "converged":
            print(f"[CG] Converged @ iter {info['iterations']}, residual norm = {info['rs']:.3e}")
        elif info["status"] == "breakdown":
            print(f"[CG] Early terminate @ iter {info['iterations']}: p^T K p not valid for SPD / NaN step.")
        else:
            print("[CG] Did not converge within max_iter.")
    u = u.to(dtype)
    return (u, info) if return_info else u


def constrained_conjugate_gradient_solver(K, elements, F, rbe2_list, spc_list, u_init=None, tol=1e-10, max_iter=1000, device="cuda:0",
                                          dtype=torch.float64, eps=1e-30, return_info=False, verbose=True):
    """CG with SPC and RBE2 constraints given as dict lists (solver.py:512-596)."""
    dev = _ops.cuda_device(device)
    return _constrained_solve(K, elements, F, parse_spc_list(spc_list, dev, torch.float64), parse_rbe2_list(rbe2_list, dev), None, u_init,
                              tol, max_iter, dev, dtype, eps, return_info, verbose)


def new_constrained_conjugate_gradient_solver(K, elements, N, rbe2_list, rbe3_list, spc_list, load_list, u_init=None, tol=1e-10,
                                              max_iter=1000, device="cuda:0", dtype=torch.float64, eps=1e-30, return_info=False,
                                              verbose=True):
    """Builds F [N,3] from the load list, then CG with SPC, RBE2 and RBE3 constraints (solver.py:702-759)."""
    dev = _ops.cuda_device(device)
    F = torch.zeros((N, 3), device=dev, dtype=torch.float64)
    apply_loads_to_F(F, load_list)
    return _constrained_solve(K, elements, F, parse_spc_list(spc_list, dev, torch.float64), parse_rbe2_list(rbe2_list, dev),
                              parse_rbe3_list(rbe3_list, dev, torch.float64), u_init, tol, max_iter, dev, dtype, eps, return_info, verbose)


def compute_diagonal_preconditioner(K, elements, N, device="cuda:0", dtype=torch.float32, fixed=None, reference_bug=False):
    """1/diag(K_global) as [N,3] without assembling K (solver.py:814-833).

    DEVIATION (documented, SURVEY.md a24): the reference's strided view `K.view(-1,nd)[:, ::nd+1]` selects COLUMN 0 of
    every row, not the diagonal, and yields a useless preconditioner.  The default here is the correct Jacobi diagonal
    (rows of `fixed` nodes set to 0); `reference_bug=True` reproduces the reference's numbers."""
    dev = _ops.cuda_device(device)
    K = torch.as_tensor(K)
    ndof = K.shape[-1] // torch.as_tensor(elements).shape[1]
    # one kernel over the node -> element incidence lists (ascending element order) instead of an index_add_ scatter
    diag = _ops.cached_plan(elements, N, dev).ebe_diag(K, ndof, dtype, col0=reference_bug)
    m = 1.0 / diag
    m[m == float("inf")] = 0.0
    if fixed is not None and not reference_bug:
        m[torch.as_tensor(fixed).to(dev).long()] = 0.0
    return m


def preconditioned_conjugate_gradient_solver(K, elements, F, M_inv, u_init=None, tol=1e-8, max_iter=1000, device="cuda:0",
                                             dtype=torch.float32, return_info=False, verbose=True, distributed=False, coords=None):
    """Textbook Jacobi-PCG exactly as the reference writes it (solver.py:766-812): z = M_inv*r, converged iff
    sqrt(r.z) < tol, no node fixing, no guards.  The loop runs in fp64 on the device; the result is cast to `dtype`.
    `distributed=True`: the multi-GPU route of stable_conjugate_gradient_solver (M_inv replicated, [N,ndof])."""
    dev = _ops.cuda_device(device)
    F = torch.as_tensor(F).to(dev)
    if distributed and _distributed_world() > 1:
        from femb200 import dist_cg
        u, info = dist_cg.solve_replicated(K, elements, F, None, u_init=u_init, tol=tol, max_iter=max_iter, eps=0.0,
                                           minv=torch.as_tensor(M_inv).reshape(F.shape), coords=coords, device=dev)
        minv = None
    else:
        minv = torch.as_tensor(M_inv).to(dev, torch.float64).reshape(-1).contiguous()
        u, info = _cg(K, elements, F, dev, mask=None, minv=minv, u_init=u_init, tol=tol, max_iter=max_iter, eps=0.0)
    if verbose:
        if info["status"] == "converged":
            print(f"Converged after {info['iterations']} iterations.")
        else:
            print("Preconditioned CG did not converge within the maximum number of iterations.")
    u = u.to(dtype)
    return (u, info) if return_info else u


def conjugate_gradient_solver_Ku(compute_Ku, R, tol=1e-8, max_iter=1000, device="cuda:0", dtype=torch.float32, return_info=False):
    """CG on an operator given as a function, K(u) delta_u = R (solver.py:1029-1065): no node fixing, no guards, start from
    zero, converged iff sqrt(r.r) < tol.  `compute_Ku` receives and returns [N,3] tensors of `dtype` on `device`, as in the
    reference; the loop itself (dot products, updates, convergence test) runs in fp64 inside libfemb200, which calls back
    for the operator once per iteration, and the result is cast to `dtype`."""
    dev = _ops.cuda_device(device)
    R = torch.as_tensor(R).to(dev)

    def apply(x):
        return compute_Ku(x.to(dtype))

    du, info = _ops.cg_solve_operator(apply, R, tol=tol, max_iter=max_iter, device=dev)
    if info["status"] != "converged":
        print("CG did not converge within the maximum number of iterations.")
    du = du.to(dtype)
    return (du, info) if return_info else du


# ------------------------------------------------------------------------------------------- modal solver

def _np_dtype(dtype):
    import numpy as np
    return np.float32 if dtype == torch.float32 else np.float64


def _invert_small_matrix(MM):
    """Gauss-Jordan without pivoting, pivots below 1e-14 replaced by 1e-14 (solver.py:1225-1243)."""
    import numpy as np
    n = MM.shape[0]
    aug = np.concatenate([MM, np.eye(n, dtype=MM.dtype)], axis=1)
    for i in range(n):
        row_i = aug[i].copy()
        pivot = row_i[i]
        if abs(pivot) < 1e-14:
            pivot = MM.dtype.type(1e-14)
        row_i = row_i / pivot
        aug[i] = row_i
        for r in range(n):
            if r != i:
                aug[r] = aug[r] - aug[r, i] * row_i
    return aug[:, n:]


def _naive_jacobi(AA, max_sweeps=30, tol=1e-10):
    """The reference's Jacobi rotations (solver.py:1245-1283) on a matrix it treats as symmetric (B^-1 A is not): largest
    off-diagonal entry, one rotation per sweep, rows rotated and then copied onto the columns.  Eigenvalues = the diagonal,
    ascending; restated step by step because the result on a non-symmetric input depends on the exact sequence."""
    import numpy as np
    n = AA.shape[0]
    ty = AA.dtype.type
    V = np.eye(n, dtype=AA.dtype)
    for _ in range(max_sweeps):
        off = AA - np.diag(np.diagonal(AA))
        idx = int(np.argmax(np.abs(off)))
        i, j = idx // n, idx % n
        if i == j:
            break
        if i > j:
            i, j = j, i
        val = AA[i, j]
        if abs(val) < tol:
            break
        theta = ty(0.5) * (AA[j, j] - AA[i, i]) / val
        t = np.sign(theta) / (abs(theta) + np.sqrt(ty(1) + theta * theta))
        c = ty(1.0) / np.sqrt(ty(1) + t * t)
        sn = t * c
        aii, aij, ajj = AA[i, i], AA[i, j], AA[j, j]
        AA[i, i] = aii - t * aij
        AA[j, j] = ajj + t * aij
        AA[i, j] = 0
        AA[j, i] = 0
        rowi, rowj = AA[i].copy(), AA[j].copy()
        AA[i] = c * rowi - sn * rowj
        AA[j] = sn * rowi + c * rowj
        AA[:, i] = AA[i].copy()
        AA[:, j] = AA[j].copy()
        Vi, Vj = V[:, i].copy(), V[:, j].copy()
        V[:, i] = c * Vi - sn * Vj
        V[:, j] = sn * Vi + c * Vj
    ev = np.diagonal(AA).copy()
    order = np.argsort(ev, kind="stable")
    return ev[order], V[:, order]


def _solve_small_gevp(A_k, B_k, npdt):
    """lam, Z of B^-1 A (solver.py:1285-1290); k x k host arithmetic in the solver's dtype."""
    A = A_k.numpy().astype(npdt)
    B = B_k.numpy().astype(npdt)
    A_ = (_invert_small_matrix(B) @ A).astype(npdt)
    return _naive_jacobi(A_.copy())


def _solve_small_gevp_sym(A_k, B_k):
    """Ritz pairs of the symmetric-definite pencil (A, B): B = L L^T, eigh(L^-1 A L^-T), Z = L^-T Q; lam ascending."""
    import numpy as np
    A = A_k.numpy().astype(np.float64)
    B = B_k.numpy().astype(np.float64)
    L = np.linalg.cholesky(0.5 * (B + B.T))
    Li = np.linalg.inv(L)
    Cm = Li @ (0.5 * (A + A.T)) @ Li.T
    lam, Q = np.linalg.eigh(0.5 * (Cm + Cm.T))
    return lam, Li.T @ Q


def _gram_schmidt_euclid(X):
    """Column-by-column Euclidean orthonormalisation exactly as the reference orders it (solver.py:1176-1199): normalise,
    subtract the projections on all previous columns at once (classical Gram-Schmidt), normalise again; columns shorter
    than 1e-14 are replaced by a unit vector."""
    for j in range(X.k):
        col = X.cols(j, j + 1)
        for stage in range(2):
            if stage == 1 and j > 0:
                prev = X.cols(0, j)
                dots = prev.gram(col)                        # [j, 1]
                prev.update_into(-dots, col, beta=1.0)      # col -= prev @ dots
            nrm = float(col.gram(col)[0, 0]) ** 0.5
            if nrm < 1e-14:
                col.data.zero_()
                if j < X.n:
                    col.data[0, j] = 1.0
            else:
                col.update_into([[1.0 / nrm]], col)
    return X


def vectorized_modal_solver(K_local, M_local, elements, rbe2_node_ids, num_nodes, num_eigs=5, max_iter=20, device="cuda:0",
                            dtype=torch.float32, X0=None, reference_gevp=False):
    """Subspace iteration on M^-1 K with a lumped mass, Euclidean Gram-Schmidt and a small generalised eigenproblem per sweep
    (solver.py:1084-1312; as written it is a block power iteration, i.e. it drifts towards the LARGEST eigenvalues of
    K u = lambda M u).  Returns (lam [num_eigs] ascending, modes [3*num_nodes, num_eigs]).

    PARITY UNPINNED: the reference raises on every input (`row_i /= pivot` divides a row by a view of itself,
    solver.py:1232-1234), and its k x k step -- Jacobi rotations for symmetric matrices applied to the non-symmetric
    B^-1 A -- does not produce eigenpairs even when that line is repaired (the restated sequence yields negative
    "eigenvalues" of an SPD pencil).  Default here: the same outer iteration with the small pencil solved as what it is,
    symmetric-definite (Cholesky of B, eigh), so lam / modes are genuine Ritz pairs; `reference_gevp=True` follows the
    reference's Gauss-Jordan + Jacobi steps literally (in `dtype`).

    The n_dof-long work runs on the device in fp64: K is assembled once (3x3 block-CSR) and applied column by column, the lumped
    mass comes from one pass over the incidence lists, and norms / projections / X^T K X / X Z are three tall-skinny kernels
    (femb_mv_*); only the k x k problems are solved on the host.  The reference
    draws its start subspace from an unseeded torch.randn; pass `X0` [3*num_nodes, num_eigs] (additive) for a reproducible run.
    For the lowest natural frequencies and mode shapes use `lowest_modes`."""
    dev = _ops.cuda_device(device)
    if not 1 <= num_eigs <= 8:
        raise ValueError("num_eigs must be between 1 and 8")
    n = num_nodes * 3
    npdt = _np_dtype(dtype)
    A = _Assembled(K_local, elements, num_nodes, 3, dev)
    plan = _ops.cached_plan(elements, num_nodes, dev)
    Mdiag = plan.ebe_diag(M_local, 3, torch.float64).reshape(-1).clamp_(min=1e-12)
    Minv = (1.0 / Mdiag).contiguous()
    mask = _dof_mask(num_nodes, 3, rbe2_node_ids, dev)
    if X0 is None:
        X0 = torch.randn(n, num_eigs, device=dev, dtype=dtype)
    X = _ops.MultiVec.from_columns(X0, dev)
    if X.n != n or X.k != num_eigs:
        raise ValueError(f"X0 must be [{n}, {num_eigs}]")

    def apply_K(V):
        out = _ops.MultiVec(torch.empty_like(V.data))
        for i in range(V.k):
            out.data[i] = A.spmv(V.data[i])
        return out

    def build_Ak_Bk(V):
        return V.gram(apply_K(V)), V.gram(V, w=Mdiag)

    def gevp(V):
        A_k, B_k = build_Ak_Bk(V)
        return _solve_small_gevp(A_k, B_k, npdt) if reference_gevp else _solve_small_gevp_sym(A_k, B_k)

    X.scale_mask(mask=mask)
    _gram_schmidt_euclid(X)
    for _ in range(max_iter):
        Y = apply_K(X).scale_mask(scale=Minv, mask=mask)
        _gram_schmidt_euclid(Y)
        lam, Z = gevp(Y)
        Y.update_into(torch.from_numpy(Z.astype("float64")), Y)
        Y.scale_mask(mask=mask)
        _gram_schmidt_euclid(Y)
        X = Y
    lam, Z = gevp(X)
    X.update_into(torch.from_numpy(Z.astype("float64")), X)
    return torch.from_numpy(lam.copy()).to(device=dev, dtype=dtype), X.columns().to(dtype)


def lowest_modes(K_local, M_local, elements, fixed, num_nodes, num_eigs=6, tol=1e-8, max_iter=2000, X0=None, device="cuda:0",
                 dtype=torch.float64, return_info=False, verbose=True):
    """Lowest eigenpairs of K x = lam M x for 3-dof solid meshes (not in the reference): LOBPCG with a Jacobi preconditioner
    (femb200/modes.py).  K_local, M_local: element matrices [M, 3 nen, 3 nen] of any solid type (a lumped mass is a diagonal
    M_local); both are assembled on one plan into 3x3 block-CSR with one block pattern.  `fixed`: node ids or a bool node mask, all
    three dofs clamped; the result is the eigenpairs of the reduced pencil (K_ff, M_ff) with zeros on the fixed dofs (with `fixed`
    empty the six rigid-body modes come out at lam = 0).  1 <= num_eigs <= 12.

    A pair has converged when |K x - lam M x| / ((|K|_1 + |lam| |M|_1) |x|) <= tol; the solve stops when the first num_eigs have,
    or after max_iter iterations with status "maxiter" (it does not raise).  X0 [3*num_nodes, num_eigs] is optional; the rest of
    the start block comes from a fixed-seed generator, so a repeated call returns bit-identical results.
    Returns (lam [num_eigs] ascending, modes [3*num_nodes, num_eigs] M-orthonormal), cast to `dtype`; with return_info also a dict
    with iterations, status, residuals, restarts (iterations that dropped the P block), freq_hz = sqrt(max(lam, 0)) / 2 pi, loop_ms."""
    from femb200 import modes
    dev = _ops.cuda_device(device)
    if not 1 <= num_eigs <= 12:
        raise ValueError("num_eigs must be between 1 and 12")
    n = 3 * num_nodes
    if X0 is not None:
        X0 = torch.as_tensor(X0).to(torch.float64).cpu().numpy()
        if X0.shape != (n, num_eigs):
            raise ValueError(f"X0 must be [{n}, {num_eigs}]")
    plan = _ops.cached_plan(elements, num_nodes, dev)
    brow, bcol = plan.pattern(1)
    K = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(K_local, 3))
    M = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(M_local, 3))
    be = modes.DeviceBackend(K, M, _dof_mask(num_nodes, 3, fixed, dev))
    lam, S, info = modes.lobpcg(be, num_eigs, tol=tol, max_iter=max_iter, X0=X0)
    if verbose:
        if info["status"] == "converged":
            print(f"LOBPCG converged after {info['iterations']} iterations ({info['restarts']} restarts).")
        else:
            print(f"LOBPCG did not converge within {max_iter} iterations; max residual {info['residuals'].max():.3e}.")
    lam = torch.from_numpy(lam).to(device=dev, dtype=dtype)
    modes_out = S[:, :num_eigs].contiguous().to(dtype)
    return (lam, modes_out, info) if return_info else (lam, modes_out)


def subdivided_lowest_modes(coords, elements, levels, fixed_fn, E, nu, rho, num_eigs=6, tol=1e-8, max_iter=500, shift=0.0, device="cuda:0",
                            dtype=torch.float64, return_info=False, verbose=True):
    """Lowest eigenpairs of K x = lam M x on a refined C3D4 mesh (not in the reference): the coarse mesh (coords, elements) is refined
    `levels` times as in hybrid_subdivided_solver, K (E, nu) and the consistent M (rho) are assembled on every level, and LOBPCG on
    the finest mesh is preconditioned by a V-cycle over the hierarchy (femb200/multigrid.py) instead of Jacobi, so the iteration
    count stays roughly flat as the mesh is refined.  fixed_fn(coords_l) -> clamped node ids (all three dofs) on every level.
    The result is what lowest_modes returns on the finest mesh, within tol (same backward-error test, M-orthonormal modes, zeros on
    fixed dofs).  `shift` >= 0: the preconditioner approximates (K + shift M)^-1; 0 suits any clamped model, a free-free model needs
    shift > 0 (a ValueError says so when the coarse K + shift M is singular).  The coarse mesh may hold at most
    multigrid.MAX_COARSE_DOFS free dofs (dense factor).  1 <= num_eigs <= 12.
    Returns (lam [num_eigs], modes [3*N_fine, num_eigs], coords_fine, elements_fine), lam and modes cast to `dtype`; with
    return_info also the dict of lowest_modes plus `levels` (nodes, tets, dofs per level, coarsest first) and `shift`."""
    from femb200 import modes, multigrid
    dev = _ops.cuda_device(device)
    if not 1 <= num_eigs <= 12:
        raise ValueError("num_eigs must be between 1 and 12")
    if not shift >= 0.0:
        raise ValueError("shift must be >= 0")
    if int(levels) != levels or levels < 0:
        raise ValueError("levels must be a non-negative integer")
    H = multigrid.Hierarchy(coords, elements, int(levels), fixed_fn, E, nu, rho, shift, dev, _el)
    lam, S, info = modes.lobpcg(multigrid.MultilevelBackend(H), num_eigs, tol=tol, max_iter=max_iter)
    info["levels"], info["shift"] = H.describe(), float(shift)
    if verbose:
        if info["status"] == "converged":
            print(f"Multigrid LOBPCG converged after {info['iterations']} iterations on {H.L[-1].n} dofs ({len(H.L)} levels).")
        else:
            print(f"Multigrid LOBPCG did not converge within {max_iter} iterations; max residual {info['residuals'].max():.3e}.")
    lam = torch.from_numpy(lam).to(device=dev, dtype=dtype)
    modes_out = S[:, :num_eigs].contiguous().to(dtype)
    out = (lam, modes_out, H.coords, H.tets)
    return out + (info,) if return_info else out


def _buckling_args(num_eigs, fixed_nodes):
    if not 1 <= num_eigs <= 12:
        raise ValueError("num_eigs must be between 1 and 12")
    f = torch.as_tensor(fixed_nodes if fixed_nodes is not None else [])
    if f.numel() == 0 or (f.dtype == torch.bool and not bool(f.any())):
        raise ValueError("no node is fixed: a free-free model has no linear buckling problem (K is singular)")


def _buckling_report(kind, info, max_iter):
    if info["status"] == "converged":
        print(f"{kind} buckling LOBPCG converged after {info['iterations']} iterations (reference solve: {info['static_iterations']} iterations).")
    else:
        print(f"{kind} buckling LOBPCG did not converge within {max_iter} iterations; max residual {info['residuals'].max():.3e}.")


def buckling_modes(coords, elements, F, fixed, E, nu, num_eigs=4, tol=1e-8, max_iter=2000, static_tol=1e-10, static_max_iter=20000,
                   integral_point=None, device="cuda:0", dtype=torch.float64, return_info=False, verbose=True):
    """Linear buckling of a C3D4 (elements [M,4]) or C3D10 ([M,10]) mesh under the reference load F [N,3] (not in the reference).
    The reference state u_ref = K^-1 F comes from the device Jacobi-PCG (|F - K u| <= static_tol |F|, else ValueError), K_G is the
    geometric stiffness of its stress, and LOBPCG with the Jacobi preconditioner of K solves K_G phi = nu K phi on the free dofs
    (femb200/buckling.py).  Load factor lam = -1/nu for nu < 0, +inf for nu >= 0 (no buckling in that pair): (K + lam K_G) phi = 0.
    `fixed`: node ids or a bool node mask, all three dofs clamped (a free-free model is refused).  C3D10 integrates K and K_G with
    `integral_point` [nq<=16, 4] rows (xi, eta, zeta, w), by default the degree-5 14-point rule (exact for straight-sided tets), not
    the reference's 11-point rule; like compute_c3d10_K_matrix it needs detJ > 0.  1 <= num_eigs <= 12; a pair has converged when |K_G x - nu K x| / ((|K_G|_1 + |nu| |K|_1) |x|)
    <= tol (max_iter reached: status "maxiter", no error).  A repeated call returns bit-identical results.
    Returns (load_factors [num_eigs] ascending, modes [3N, num_eigs] K-orthonormal with zeros on fixed dofs, u_ref [N,3]) cast to
    `dtype`; with return_info also the dict of lowest_modes without freq_hz, plus nu (the pencil's eigenvalues) and
    static_iterations / static_residual of the reference solve."""
    from femb200 import buckling
    dev = _ops.cuda_device(device)
    elements = _ops.index(elements, dev)
    if elements.dim() != 2 or elements.shape[1] not in (4, 10):
        raise ValueError(f"elements must be [M,4] (C3D4) or [M,10] (C3D10), got {tuple(elements.shape)}")
    _buckling_args(num_eigs, fixed)
    coords = _ops.real(coords, dev, torch.float64)
    N = coords.shape[0]
    mask = _dof_mask(N, 3, fixed, dev)
    plan = _ops.CsrPlan(elements, N, dev)
    brow, bcol = plan.pattern(1)
    if elements.shape[1] == 4:
        Ke = _el.compute_c3d4_K_matrix(coords, elements, E, nu, device=dev, dtype=torch.float64)
    else:
        rule = torch.tensor(_el._exact_pts(_ops.C3D10, integral_point, torch.float64), dtype=torch.float64)
        Ke = _el.compute_c3d10_K_matrix(coords, elements, E, nu, integral_point=rule, device=dev, dtype=torch.float64)
    K = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ke, 3))
    del Ke
    u, static_its, static_res = buckling.static_jacobi(K, mask, F, static_tol, static_max_iter)
    u = u.reshape(N, 3)
    if elements.shape[1] == 4:
        KGe = _el.compute_c3d4_KG_matrix(coords, elements, u, E, nu, device=dev, dtype=torch.float64)
    else:
        KGe = _el.compute_c3d10_KG_matrix(coords, elements, u, E, nu, integral_point=rule, device=dev, dtype=torch.float64)
    KG = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(KGe, 3))
    del KGe
    lam, modes_out, info = buckling.solve(buckling.JacobiBackend(KG, K, mask), num_eigs, tol, max_iter)
    info["static_iterations"], info["static_residual"] = static_its, static_res
    if verbose:
        _buckling_report("Jacobi", info, max_iter)
    out = (torch.from_numpy(lam).to(device=dev, dtype=dtype), modes_out.contiguous().to(dtype), u.to(dtype))
    return out + (info,) if return_info else out


def subdivided_buckling_modes(coords, elements, levels, load_fn, fixed_fn, E, nu, num_eigs=4, tol=1e-8, max_iter=500, static_tol=1e-10,
                              static_max_iter=500, device="cuda:0", dtype=torch.float64, return_info=False, verbose=True):
    """Linear buckling on a refined C3D4 mesh (not in the reference): the coarse mesh (coords, elements [M,4]) is refined `levels` times
    as in subdivided_lowest_modes, load_fn(coords_l, tets_l) -> F [N_l, 3] gives the reference load on the finest mesh and
    fixed_fn(coords_l) the clamped node ids on every level.  What buckling_modes computes on the finest mesh, with the Jacobi
    preconditioner replaced by one V-cycle over the hierarchy (femb200/multigrid.py at shift 0) in both the reference solve (PCG) and
    LOBPCG, so the iteration counts stay roughly flat as the mesh is refined.  No mass is assembled.  The coarse mesh may hold at most
    multigrid.MAX_COARSE_DOFS free dofs.  Returns (load_factors, modes, u_ref, coords_fine, elements_fine) (+ info, which also holds
    `levels`: nodes, tets, dofs per level, coarsest first)."""
    from femb200 import buckling, multigrid
    dev = _ops.cuda_device(device)
    elements = _ops.index(elements, dev)
    if elements.dim() != 2 or elements.shape[1] != 4:
        raise ValueError(f"subdivided_buckling_modes refines C3D4 meshes: elements must be [M,4], got {tuple(elements.shape)}")
    if int(levels) != levels or levels < 0:
        raise ValueError("levels must be a non-negative integer")
    coords = _ops.real(coords, dev, torch.float64)
    _buckling_args(num_eigs, fixed_fn(coords))
    H = multigrid.Hierarchy(coords, elements, int(levels), fixed_fn, E, nu, None, 0.0, dev, _el)
    top = H.L[-1]
    u, static_its, static_res = buckling.static_multigrid(H, load_fn(H.coords, H.tets), static_tol, static_max_iter)
    u = u.reshape(-1, 3)
    KGe = _el.compute_c3d4_KG_matrix(H.coords, H.tets, u, E, nu, device=dev, dtype=torch.float64)
    brow, bcol = top.plan.pattern(1)
    KG = _ops.Bsr3.from_csr_values(brow, bcol, top.plan.assemble(KGe, 3))
    del KGe
    lam, modes_out, info = buckling.solve(buckling.MultilevelBackend(H, KG), num_eigs, tol, max_iter)
    info["static_iterations"], info["static_residual"], info["levels"] = static_its, static_res, H.describe()
    if verbose:
        _buckling_report("Multigrid", info, max_iter)
    out = (torch.from_numpy(lam).to(device=dev, dtype=dtype), modes_out.contiguous().to(dtype), u.to(dtype), H.coords, H.tets)
    return out + (info,) if return_info else out


def amg_lowest_modes(coords, K_local, M_local, elements, fixed, num_eigs=6, tol=1e-8, max_iter=500, shift=0.0, device="cuda:0",
                     dtype=torch.float64, return_info=False, verbose=True):
    """Lowest eigenpairs of K x = lam M x for any 3-dof solid mesh (not in the reference), as lowest_modes computes them, with LOBPCG
    preconditioned by one V-cycle of smoothed-aggregation algebraic multigrid (femb200/amg.py) instead of Jacobi: the hierarchy is
    built on the device from the assembled operator and the node coordinates [N, 3], so no mesh hierarchy is needed and the
    iteration count stays roughly flat as the mesh is refined.  K_local, M_local, elements, fixed: as lowest_modes (K and M are
    assembled on one plan).  `shift` >= 0: the cycle approximates (K + shift M)^-1; a free-free model needs shift > 0 (a ValueError
    says so).  Returns what lowest_modes returns; info also holds `levels` (nodes, dofs, free dofs, nnzb per level, coarsest first),
    `operator_complexity` and `setup_ms` (aggregation, tentative, lambda, spgemm, factor)."""
    from femb200 import amg, modes, multigrid
    dev = _ops.cuda_device(device)
    if not 1 <= num_eigs <= 12:
        raise ValueError("num_eigs must be between 1 and 12")
    if not shift >= 0.0:
        raise ValueError("shift must be >= 0")
    coords = _ops.real(coords, dev, torch.float64)
    N = coords.shape[0]
    plan = _ops.cached_plan(elements, N, dev)
    brow, bcol = plan.pattern(1)
    K = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(K_local, 3))
    M = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(M_local, 3))
    A = K if not shift else _ops.Bsr3(brow, bcol, K.bval + float(shift) * M.bval)
    H = amg.AmgHierarchy(A, _dof_mask(N, 3, fixed, dev), coords, K=K, M=M)
    lam, S, info = modes.lobpcg(multigrid.MultilevelBackend(H), num_eigs, tol=tol, max_iter=max_iter)
    d = H.describe()
    info["levels"], info["operator_complexity"], info["setup_ms"], info["shift"] = d["levels"], d["operator_complexity"], d["setup_ms"], float(shift)
    if verbose:
        if info["status"] == "converged":
            print(f"AMG LOBPCG converged after {info['iterations']} iterations on {3 * N} dofs ({len(H.L)} levels).")
        else:
            print(f"AMG LOBPCG did not converge within {max_iter} iterations; max residual {info['residuals'].max():.3e}.")
    lam = torch.from_numpy(lam).to(device=dev, dtype=dtype)
    modes_out = S[:, :num_eigs].contiguous().to(dtype)
    return (lam, modes_out, info) if return_info else (lam, modes_out)


def amg_buckling_modes(coords, elements, F, fixed, E, nu, num_eigs=4, tol=1e-8, max_iter=500, static_tol=1e-10, static_max_iter=500,
                       integral_point=None, device="cuda:0", dtype=torch.float64, return_info=False, verbose=True):
    """Linear buckling of a C3D4 or C3D10 mesh (not in the reference): what buckling_modes computes, with the Jacobi preconditioner
    replaced by one V-cycle of smoothed-aggregation algebraic multigrid (femb200/amg.py, built from K and the coordinates) in both
    the reference solve (PCG, buckling.static_multigrid) and LOBPCG.  Arguments, refusals and returns as buckling_modes; info also
    holds `levels`, `operator_complexity` and `setup_ms` of the hierarchy."""
    from femb200 import amg, buckling
    dev = _ops.cuda_device(device)
    elements = _ops.index(elements, dev)
    if elements.dim() != 2 or elements.shape[1] not in (4, 10):
        raise ValueError(f"elements must be [M,4] (C3D4) or [M,10] (C3D10), got {tuple(elements.shape)}")
    _buckling_args(num_eigs, fixed)
    coords = _ops.real(coords, dev, torch.float64)
    N = coords.shape[0]
    mask = _dof_mask(N, 3, fixed, dev)
    plan = _ops.CsrPlan(elements, N, dev)
    brow, bcol = plan.pattern(1)
    if elements.shape[1] == 4:
        Ke = _el.compute_c3d4_K_matrix(coords, elements, E, nu, device=dev, dtype=torch.float64)
    else:
        rule = torch.tensor(_el._exact_pts(_ops.C3D10, integral_point, torch.float64), dtype=torch.float64)
        Ke = _el.compute_c3d10_K_matrix(coords, elements, E, nu, integral_point=rule, device=dev, dtype=torch.float64)
    K = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ke, 3))
    del Ke
    H = amg.AmgHierarchy(K, mask, coords, K=K)
    u, static_its, static_res = buckling.static_multigrid(H, F, static_tol, static_max_iter)
    u = u.reshape(N, 3)
    if elements.shape[1] == 4:
        KGe = _el.compute_c3d4_KG_matrix(coords, elements, u, E, nu, device=dev, dtype=torch.float64)
    else:
        KGe = _el.compute_c3d10_KG_matrix(coords, elements, u, E, nu, integral_point=rule, device=dev, dtype=torch.float64)
    KG = _ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(KGe, 3))
    del KGe
    lam, modes_out, info = buckling.solve(buckling.MultilevelBackend(H, KG), num_eigs, tol, max_iter)
    d = H.describe()
    info["static_iterations"], info["static_residual"] = static_its, static_res
    info["levels"], info["operator_complexity"], info["setup_ms"] = d["levels"], d["operator_complexity"], d["setup_ms"]
    if verbose:
        _buckling_report("AMG", info, max_iter)
    out = (torch.from_numpy(lam).to(device=dev, dtype=dtype), modes_out.contiguous().to(dtype), u.to(dtype))
    return out + (info,) if return_info else out


def static_structure_solver(coords, force, fixed, c3d4=None, c3d6=None, c3d8=None, s3=None, s4=None, material=None, u_init=None,
                            tol=1e-10, max_iter=1000, device="cuda:0", dtype=torch.float64, eps=1e-30, return_info=False, verbose=True):
    """Mixed-element static solve on [N,6] (solver.py:11-135): solids act on the translations, shells on all six dofs
    in their own frames.  Every element family is brought to global 6-dof element matrices and assembled into ONE CSR
    (padded connectivity is avoided by assembling each family on its own plan and summing the CSR triplets)."""
    dev = _ops.cuda_device(device)
    coords = torch.as_tensor(coords).to(dev, torch.float64)
    force = torch.as_tensor(force).to(dev, torch.float64)
    N = coords.shape[0]
    E, nu = (material or {}).get("E"), (material or {}).get("nu")
    fams = []

    def solid6(K3):
        M, nd, _ = K3.shape
        nen = nd // 3
        K6 = torch.zeros((M, nen, 6, nen, 6), device=dev, dtype=torch.float64)
        K6[:, :, :3, :, :3] = K3.reshape(M, nen, 3, nen, 3)
        return K6.reshape(M, nen * 6, nen * 6)

    if c3d4 is not None:
        fams.append((solid6(_el.compute_c3d4_K_matrix(coords, c3d4, E, nu, device=dev, dtype=torch.float64)), c3d4))
    if c3d8 is not None:
        fams.append((solid6(_el.compute_c3d8_K_matrix(coords, c3d8, E, nu, device=dev, dtype=torch.float64)), c3d8))
    if c3d6 is not None:
        fams.append((solid6(_el.compute_c3d6_K_matrix(coords, c3d6, E, nu, device=dev, dtype=torch.float64)), c3d6))
    if s3 is not None:
        K = _sh.compute_s3_K_matrix(coords, s3, material["membrane"], material["bending"], device=dev, dtype=torch.float64)
        fams.append((_shell_global_K(K, _sh.compute_s3_local_unitvector(coords, s3, device=dev)), s3))
    if s4 is not None:
        K = _sh.compute_s4_K_matrix(coords, s4, material["membrane"], material["bending"], device=dev, dtype=torch.float64)
        fams.append((_shell_global_K(K, _sh.compute_s4_local_unitvector(coords, s4, device=dev)), s4))
    if verbose:
        print("Preprocessing done.")
    mats = []
    for K6, conn in fams:
        crow, col, val, _ = _operator(K6, torch.as_tensor(conn).to(dev), N, dev)
        mats.append((crow, col, val))
    u, info = _ops.cg_solve_multi(mats, force, mask=_dof_mask(N, 6, fixed, dev), u_init=u_init, tol=tol, max_iter=max_iter, eps=eps)
    if verbose:
        _report("CG", info, max_iter)
    u = u.to(dtype)
    return (u, info) if return_info else u


def hybrid_subdivided_solver(coords, elements, levels, load_fn, fixed_fn, E=None, nu=None, kind="elasticity", tol=1e-8, max_iter=10000,
                             device="cuda:0", verbose=True, mode="multilevel"):
    """Additive API for the reference's announced "hybrid solver of iterative and inverse methods with sub-divided mesh"
    (README.md:7; the notebook stops before any solve loop): the coarse C3D4 mesh is solved directly (dense Cholesky) and
    refined `levels` times (c3d4_to_c3d10 + c3d10_to_c3d4).  mode="multilevel": CG on the finest mesh preconditioned by a
    V-cycle over the hierarchy with the direct solve at the bottom; mode="cascade": every level solved by the reference CG
    loop warm-started from the prolongated coarser solution.  See femb200/hybrid.py.
    Returns (u_fine, coords_fine, elements_fine, info)."""
    from femb200 import hybrid
    return hybrid.hybrid_solve(coords, elements, levels, load_fn, fixed_fn, E, nu, kind, tol, max_iter, device, _el, verbose, mode)
