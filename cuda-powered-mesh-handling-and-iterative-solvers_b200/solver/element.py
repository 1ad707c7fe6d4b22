"""Drop-in mirror of the reference's `solver/element.py` function API on hand-written sm_100a kernels.

Use exactly like the reference (`sys.path.append(<this dir>); import element`): same function names,
positional order, defaults (device="cuda:0", dtype=torch.float32) and return shapes; tensors in and
out stay on the device.  Every function is a thin wrapper that allocates outputs with torch and calls
libfemb200 through ctypes (femb200/ops.py); there is no CPU path and no torch op chain behind them.
Each docstring names the reference lines it replaces (paths relative to the reference's solver/).

Deliberately reproduced quirks (SURVEY.md section 8a): the type dispatchers drop `dtype` (q2), C3D6 and S4
quadrature constants are fp32-rounded (q1), detJ is signed (q3), C3D10/C3D6 weights are the reference's (q4),
shared-face pairs are emitted lower-element-first (the reference's order is implementation-defined, q5).
"""
from __future__ import annotations

import os
import sys

import torch

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if _PKG not in sys.path:
    sys.path.insert(0, _PKG)

from femb200 import ops as _ops  # noqa: E402
from femb200.ops import CsrPlan  # noqa: E402,F401


def _pts(kind, integral_point, dtype, single_point=False):
    """Resolve quadrature input to a host list of [xi,eta,zeta,w] rows, rounded through `dtype` as the reference does."""
    if integral_point is None:
        rows = torch.tensor(_ops.default_points(kind), dtype=torch.float64)
    else:
        ip = torch.as_tensor(integral_point).detach().to("cpu")
        if single_point:
            ip = torch.cat([ip.reshape(3).to(torch.float64), torch.ones(1, dtype=torch.float64)]).reshape(1, 4)
        rows = torch.stack([ip[:, 0], ip[:, 1], ip[:, 2], ip[:, -1]], dim=1)
    return rows.to(dtype).to(torch.float64).tolist()


def human_readable_number(num):
    """'12.3M'-style counts for the notebooks' prints (element.py:23-37): one decimal, suffix K / M / B / T / Quad / Quint."""
    for power, suffix in ((18, "Quint"), (15, "Quad"), (12, "T"), (9, "B"), (6, "M"), (3, "K")):
        if abs(num) >= 10 ** power:
            return f"{num / 10 ** power:.1f}{suffix}"
    return f"{num:.1f}"


# ------------------------------------------------------------------------------------------- constants

def compute_elasticity_matrix(E, nu, device="cuda:0", dtype=torch.float32):
    """Isotropic 6x6 D in Voigt order xx,yy,zz,xy,yz,zx (reference element.py:282-306)."""
    c = E / ((1 + nu) * (1 - 2 * nu))
    s = (1 - 2 * nu) / 2
    rows = [[1 - nu, nu, nu, 0, 0, 0], [nu, 1 - nu, nu, 0, 0, 0], [nu, nu, 1 - nu, 0, 0, 0],
            [0, 0, 0, s, 0, 0], [0, 0, 0, 0, s, 0], [0, 0, 0, 0, 0, s]]
    return c * torch.tensor(rows, device=device, dtype=dtype)


# ------------------------------------------------------------------------------------------- dispatchers

def to_c3d4(elements, device="cuda:0"):
    """element.py:355-364"""
    n = elements.shape[1]
    if n == 6:
        return c3d6_to_c3d4(elements, device)
    if n == 8:
        return c3d8_to_c3d4(elements, device)
    if n == 10:
        return c3d10_to_c3d4(elements, device)
    return None   # the reference's dispatcher does not route C3D20 either; call c3d20_to_c3d4 directly


def to_2nd_order(coords, elements, rbe2=None, rbe3=None, device="cuda:0", dtype=torch.float32):
    """element.py:366-369"""
    if elements.shape[1] == 4:
        return c3d4_to_c3d10(coords, elements, rbe2, rbe3, dtype=dtype)
    return None


def _unsupported(element_type):
    raise ValueError(f"Unsupported element type: {element_type}")


def integral_points(element_type, device="cuda:0"):
    """element.py:371-378 -- always float32 (the dispatcher drops dtype, quirk q2)."""
    t = element_type.lower()
    fn = {"c3d8": c3d8_integration_points, "c3d10": c3d10_integration_points, "c3d6": c3d6_integration_points,
          "c3d20": c3d20_integration_points, "c3d15": c3d15_integration_points}.get(t)
    return fn(device) if fn else _unsupported(element_type)


def compute_Jacobian(coords, elements, element_type, integral_point=None, device="cuda:0"):
    """element.py:380-388 (float32 result, q2; 'c3d8i' aliases C3D8 here only)."""
    t = element_type.lower()
    fn = {"c3d8": compute_c3d8_Jacobian, "c3d8i": compute_c3d8_Jacobian, "c3d10": compute_c3d10_Jacobian,
          "c3d6": compute_c3d6_Jacobian, "c3d20": compute_c3d20_Jacobian, "c3d15": compute_c3d15_Jacobian}.get(t)
    return fn(coords, elements, integral_point, device) if fn else _unsupported(element_type)


def compute_shape_gradients(coords, elements, element_type, integral_point=None, device="cuda:0"):
    """element.py:390-397 (float32 result, q2)."""
    t = element_type.lower()
    fn = {"c3d8": compute_c3d8_shape_gradients, "c3d10": compute_c3d10_shape_gradients, "c3d6": compute_c3d6_shape_gradients,
          "c3d20": compute_c3d20_shape_gradients, "c3d15": compute_c3d15_shape_gradients}.get(t)
    return fn(coords, elements, integral_point, device) if fn else _unsupported(element_type)


def compute_B_matrix(coords, elements, integral_point, element_type, device="cuda:0", dtype=torch.float32):
    """element.py:399-407 (dtype honoured for C3D4 only, q2)."""
    t = element_type.lower()
    if t == "c3d4":
        return compute_c3d4_B_matrix(coords, elements, device, dtype)
    fn = {"c3d8": compute_c3d8_B_matrix, "c3d10": compute_c3d10_B_matrix, "c3d6": compute_c3d6_B_matrix,
          "c3d20": compute_c3d20_B_matrix, "c3d15": compute_c3d15_B_matrix}.get(t)
    return fn(coords, elements, integral_point, device) if fn else _unsupported(element_type)


def compute_K_matrix(coords, elements, element_type, E, nu, integral_point=None, single=True, device="cuda:0", dtype=torch.float32):
    """element.py:419-427"""
    t = element_type.lower()
    if t == "c3d4":
        return compute_c3d4_K_matrix(coords, elements, E, nu, device, dtype)
    fn = {"c3d8": compute_c3d8_K_matrix, "c3d10": compute_c3d10_K_matrix, "c3d6": compute_c3d6_K_matrix,
          "c3d20": compute_c3d20_K_matrix, "c3d15": compute_c3d15_K_matrix}.get(t)
    return fn(coords, elements, E, nu, integral_point, single, device, dtype) if fn else _unsupported(element_type)


def compute_element_stress(coords, elements, displacement, E, nu, element_type, integral_point=None, single=True, device="cuda:0",
                           dtype=torch.float32):
    """element.py:409-417"""
    t = element_type.lower()
    if t == "c3d4":
        return compute_c3d4_element_stress(coords, elements, displacement, E, nu, device, dtype)
    fn = {"c3d8": compute_c3d8_element_stress, "c3d10": compute_c3d10_element_stress, "c3d6": compute_c3d6_element_stress,
          "c3d20": compute_c3d20_element_stress, "c3d15": compute_c3d15_element_stress}.get(t)
    return fn(coords, elements, displacement, E, nu, integral_point, single, device, dtype) if fn else _unsupported(element_type)


def compute_M_matrix(coords, elements, element_type, rho, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Consistent mass [M,nd,nd] by element type.  Additive: the reference only calls an undefined
    compute_c3d4_M_matrix (solver_example.ipynb cell 13) -- parity unpinned, see compute_c3d10_M_matrix."""
    t = element_type.lower()
    if t == "c3d4":
        return compute_c3d4_M_matrix(coords, elements, rho, device, dtype)
    kind = {"c3d8": _ops.C3D8, "c3d10": _ops.C3D10, "c3d6": _ops.C3D6, "c3d20": _ops.C3D20, "c3d15": _ops.C3D15}.get(t)
    return _solid_M(kind, coords, elements, rho, integral_point, device, dtype) if kind else _unsupported(element_type)


# ------------------------------------------------------------------------------------------- stress helpers

def compute_stress_tensor(stress_vector):
    """Voigt [M,6] (xx,yy,zz,xy,yz,zx) -> [M,3,3] on the tensor's own device and dtype (element.py:308-330)."""
    return _ops.stress_helper(0, stress_vector)


def compute_von_mises_stress(stress_tensor):
    """[M,3,3] -> [M] (element.py:332-353)."""
    return _ops.stress_helper(1, stress_tensor)


def compute_node_vm_stress(coords, elements, element_vm_stress, device="cuda:0", dtype=torch.float32):
    """Node value = mean over the elements containing the node (element.py:466-504); the reference scatters with atomic
    index_add, here each node sums its incidence list in ascending element order (deterministic)."""
    dev = _ops.cuda_device(device)
    plan = _ops.cached_plan(elements, torch.as_tensor(coords).shape[0], dev)
    return plan.node_average(element_vm_stress, dtype)


def _stress(kind, coords, elements, displacement, E, nu, integral_point, single, device, dtype, point_major):
    pts = _pts(kind, integral_point, dtype)
    S, V = _ops.solid_stress(kind, coords, elements, displacement, pts, E, nu, single, device, dtype)
    if single or point_major:
        return S, V
    return S.permute(1, 0, 2, 3).contiguous(), V.t().contiguous()


def compute_nodal_forces(K, elements, displacement, device="cuda:0", dtype=torch.float32):
    """Matrix-free y = K u (element.py:429-464).  Instead of gather -> bmm -> atomic index_add, one thread per dof row
    walks the node's incidence list in ascending element order (deterministic).  The incidence plan of `elements` is
    cached across calls (the reference rebuilds its dof table on every call)."""
    dev = _ops.cuda_device(device)
    u = _ops.real(displacement, dev, dtype)
    N, ndof = u.shape
    plan = _ops.cached_plan(elements, N, dev)
    return plan.ebe_apply(K, u, ndof, None, dtype)


# ------------------------------------------------------------------------------------------- tetrahedra

def compute_tetrahedral_volumes(coords, elements, device="cuda:0", dtype=torch.float32):
    """|det[v1,v2,v3]|/6 (element.py:514-541)."""
    return _ops.volumes(_ops.C3D4, coords, elements, device, dtype)


def compute_tetrahedral_surface_faces_with_fourth_node(elements, device="cuda:0"):
    """Faces that occur once, slot-major order, plus the off-face node (element.py:543-579)."""
    f, x, _ = _ops.entities(_ops.ENT_TET_FACES, elements, device, want_shared=False)
    return f, x


def compute_tetrahdral_surface_normals(coords, elements, device="cuda:0", dtype=torch.float32):
    """Outward unit normals of the surface faces (element.py:581-619)."""
    f, x = compute_tetrahedral_surface_faces_with_fourth_node(elements, device)
    return _ops.surface_normals(coords, f, x, 2, device, dtype)


def compute_tetrahedral_normals_and_area(coords, elements, device="cuda:0", dtype=torch.float32):
    """[M,4,3] area-weighted outward face normals (element.py:652-705)."""
    return _ops.face_normals_area(_ops.C3D4, coords, elements, device, dtype)


def identify_tetrahedral_shared_faces(elements, device="cuda:0"):
    """[S,2,2] = ((elem,face),(elem,face)), rows lexicographic by sorted node triple (element.py:707-762)."""
    return _ops.entities(_ops.ENT_TET_FACES, elements, device, want_surface=False)[2]


def c3d4_to_c3d10(coords, elements, rbe2_ids=None, rbe3_ids=None, dtype=torch.float32, device=None):
    """Mid-edge insertion with the reference's first-encounter numbering (element.py:777-833) as device kernels
    (csrc/refine.cu: one stable radix sort of the edge keys, a max-scan of the group heads, a prefix sum over the first
    occurrences) instead of a Python dict loop: an edge's new id is N + (rank of its first occurrence in element-major,
    slot (0,1),(1,2),(2,0),(0,3),(1,3),(2,3) order).  Returns (coords', elems[int32], rbe2', rbe3') on the CPU like the
    reference unless `device` is given.  Mid points are formed in the precision of `coords` (the reference uses Python
    floats, i.e. fp64, for fp64 input) and then cast to `dtype`."""
    dev = torch.as_tensor(elements).device if device is None else torch.device(device)
    work = dev if dev.type == "cuda" else torch.device("cuda:0")
    x = torch.as_tensor(coords)
    N = x.shape[0]
    new_coords, new_elems, edges = _ops.p1_to_p2(x, elements, work, dtype)

    def grow(ids):
        if ids is None:
            return torch.tensor([], dtype=torch.int32)
        m = torch.zeros(N, dtype=torch.bool, device=work)
        m[torch.as_tensor(ids).to(work).long()] = True
        both = m[edges[:, 0].long()] & m[edges[:, 1].long()]
        return torch.cat([torch.nonzero(m).reshape(-1), N + torch.nonzero(both).reshape(-1)]).to(torch.int32)

    out_dev = torch.device("cpu") if device is None else dev
    return new_coords.to(out_dev), new_elems.to(out_dev), grow(rbe2_ids).to(out_dev), grow(rbe3_ids).to(out_dev)


def compute_c3d4_B_matrix(coords, elements, device="cuda:0", dtype=torch.float32):
    """[M,6,12]; raises ValueError when any |det[1,x,y,z]| < 1e-12 (element.py:835-881)."""
    return _ops.c3d4(1, coords, elements, device=device, dtype=dtype)


def compute_c3d4_shape_gradients(coords, elements, device="cuda:0", dtype=torch.float32):
    """[M,4,3] P1 gradients (the `grads` of element.py:862-866; additive helper)."""
    return _ops.c3d4(0, coords, elements, device=device, dtype=dtype)


def compute_c3d4_K_matrix(coords, elements, E, nu, device="cuda:0", dtype=torch.float32, out=None):
    """K = B^T D B V, [M,12,12] (element.py:883-903).  `out=` (additive): write into a caller-owned buffer."""
    return _ops.c3d4(2, coords, elements, E, nu, device, dtype, out=out)


def compute_c3d4_poisson_K_matrix(coords, elements, device="cuda:0", dtype=torch.float32, out=None):
    """Scalar Laplace stiffness V G G^T [M,4,4].  Not in the reference (parity unpinned); additive."""
    return _ops.c3d4(3, coords, elements, device=device, dtype=dtype, out=out)


def compute_c3d4_M_matrix(coords, elements, rho, device="cuda:0", dtype=torch.float32):
    """Consistent mass [M,12,12].  Called by the reference's notebook but defined nowhere (parity unpinned)."""
    return _ops.c3d4(4, coords, elements, rho, 0.0, device, dtype)


def compute_c3d4_element_stress(coords, elements, displacement, E, nu, device="cuda:0", dtype=torch.float32):
    """([M,3,3], [M]) constant-strain stress and von Mises (element.py:905-939)."""
    return _ops.solid_stress(_ops.C3D4, coords, elements, displacement, [[0.25, 0.25, 0.25, 1.0]], E, nu, True, device, dtype)


def compute_c3d4_KG_matrix(coords, elements, displacement, E, nu, device="cuda:0", dtype=torch.float32):
    """Geometric stiffness [M,12,12] of the constant stress of `displacement` [N,3]: block (a,b) = V g_a^T sigma g_b I3.
    Not in the reference (parity unpinned); the initial-stress matrix of linear buckling (solver.buckling_modes)."""
    return _ops.solid_geometric(_ops.C3D4, coords, elements, displacement, [[0.25, 0.25, 0.25, 1.0]], E, nu, device, dtype)


def c3d10_to_c3d4(c3d10_elements, device="cuda:0"):
    """8 children per C3D10 (element.py:963-993)."""
    return _ops.to_c3d4(_ops.C3D10, c3d10_elements, device)


def _points_out(kind, device, dtype):
    rows = torch.tensor(_ops.default_points(kind), dtype=torch.float64)
    return rows[:, :3].to(dtype).to(device), rows[:, 3].to(dtype).to(device)


def c3d10_integration_points(device="cuda:0", dtype=torch.float32):
    """The reference's 11-point rule, weights summing to 0.45 (element.py:995-1024)."""
    return _points_out(_ops.C3D10, device, dtype)


def _solid(kind, what, coords, elements, integral_point, device, dtype, E=0.0, nu=0.0, single_point=True, out=None):
    pts = _pts(kind, integral_point, dtype, single_point=single_point)
    return _ops.solid(kind, what, coords, elements, pts, E, nu, device, dtype, out=out)


def _solid_K(kind, coords, elements, E, nu, integral_point, single, device, dtype, out=None):
    return _solid(kind, 3 if single else 4, coords, elements, integral_point, device, dtype, E, nu, single_point=False, out=out)


def _exact_pts(kind, integral_point, dtype):
    """The rule of the operators that are not in the reference (mass, geometric stiffness): the caller's points, or by default
    femb_mass_points (for C3D10 the degree-5 14-point rule, not the reference's 11-point rule whose weights sum to 0.45)."""
    if integral_point is None:
        return torch.tensor(_ops.mass_points(kind), dtype=torch.float64).to(dtype).to(torch.float64).tolist()
    return _pts(kind, integral_point, dtype)


def _solid_M(kind, coords, elements, rho, integral_point, device, dtype):
    return _ops.solid(kind, 6, coords, elements, _exact_pts(kind, integral_point, dtype), rho, 0.0, device, dtype)


def compute_c3d10_Jacobian(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """[M,3,3] (element.py:1026-1060)."""
    return _solid(_ops.C3D10, 0, coords, elements, integral_point, device, dtype)


def compute_c3d10_shape_gradients(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """[M,10,3] (element.py:1062-1095)."""
    return _solid(_ops.C3D10, 1, coords, elements, integral_point, device, dtype)


def compute_c3d10_B_matrix(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """[M,6,30] (element.py:1097-1125)."""
    return _solid(_ops.C3D10, 2, coords, elements, integral_point, device, dtype)


def compute_c3d10_K_matrix(coords, elements, E, nu, integral_point=None, single=True, device="cuda:0", dtype=torch.float32, out=None):
    """sum_q w_q detJ_q B^T D B with signed detJ; single=False -> [n_int,M,30,30] unweighted (element.py:1191-1239).
    `out=` (additive): write into a caller-owned buffer."""
    return _solid_K(_ops.C3D10, coords, elements, E, nu, integral_point, single, device, dtype, out=out)


def compute_c3d10_element_stress(coords, elements, displacement, E, nu, integral_point=None, single=True, device="cuda:0",
                                 dtype=torch.float32):
    """single=True: ([M,3,3],[M]) weighted with the rule's weights (which sum to 0.45, q4); single=False:
    ([n_int,M,3,3],[n_int,M]) (element.py:1127-1189)."""
    return _stress(_ops.C3D10, coords, elements, displacement, E, nu, integral_point, single, device, dtype, True)


def compute_c3d10_KG_matrix(coords, elements, displacement, E, nu, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Geometric stiffness sum_q w_q |detJ_q| g_a^T sigma_q g_b I3, [M,30,30], of the stress of `displacement` [N,3]; default
    rule = degree-5 14-point (exact for straight-sided tets), integral_point [nq<=16, 4] rows (xi, eta, zeta, w) otherwise.
    Not in the reference -- parity unpinned."""
    return _ops.solid_geometric(_ops.C3D10, coords, elements, displacement, _exact_pts(_ops.C3D10, integral_point, dtype), E, nu,
                                device, dtype)


def compute_c3d10_M_matrix(coords, elements, rho, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Consistent mass rho sum_q w_q |detJ_q| N^T N (x) I3, [M,30,30]; default rule = degree-5 14-point (exact for
    straight-sided tets).  Not in the reference -- parity unpinned."""
    return _solid_M(_ops.C3D10, coords, elements, rho, integral_point, device, dtype)


# ------------------------------------------------------------------------------------------- hexahedra

def compute_hexahedral_volumes(coords, elements, device="cuda:0", dtype=torch.float32):
    """Sum of six |tet| volumes with the reference's table (element.py:1248-1291)."""
    return _ops.volumes(_ops.C3D8, coords, elements, device, dtype)


def compute_hexahedral_surface_faces_with_extra_node(elements, device="cuda:0"):
    """element.py:1293-1334 (works on [M,20] too: corner columns only)."""
    f, x, _ = _ops.entities(_ops.ENT_HEX_FACES, elements, device, want_shared=False)
    return f, x


def compute_hexahedral_surface_normals(coords, elements, device="cuda:0", dtype=torch.float32):
    """element.py:1336-1374"""
    f, x = compute_hexahedral_surface_faces_with_extra_node(elements, device)
    return _ops.surface_normals(coords, f, x, 2, device, dtype)


def compute_hexahedral_normals_and_area(coords, elements, device="cuda:0", dtype=torch.float32):
    """[M,6,3] cross(e01,e03), oriented with the element routine's own off-face table (element.py:1418-1472)."""
    return _ops.face_normals_area(_ops.C3D8, coords, elements, device, dtype)


def identify_hexahedral_shared_faces(elements, device="cuda:0"):
    """element.py:1474-1532"""
    return _ops.entities(_ops.ENT_HEX_FACES, elements, device, want_surface=False)[2]


def c3d8_to_c3d4(c3d8_elements, device="cuda:0"):
    """The reference's 6-tet table, reproduced as is although it is not a partition of the hex (element.py:1555-1581)."""
    return _ops.to_c3d4(_ops.C3D8, c3d8_elements, device)


def c3d8_integration_points(device="cuda:0", dtype=torch.float32):
    """2x2x2 Gauss, xi slowest (element.py:1583-1599)."""
    return _points_out(_ops.C3D8, device, dtype)


def compute_c3d8_Jacobian(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """element.py:1601-1632"""
    return _solid(_ops.C3D8, 0, coords, elements, integral_point, device, dtype)


def compute_c3d8_shape_gradients(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """element.py:1634-1664"""
    return _solid(_ops.C3D8, 1, coords, elements, integral_point, device, dtype)


def compute_c3d8_B_matrix(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """element.py:1666-1694"""
    return _solid(_ops.C3D8, 2, coords, elements, integral_point, device, dtype)


def compute_c3d8_K_matrix(coords, elements, E, nu, integral_point=None, single=True, device="cuda:0", dtype=torch.float32):
    """element.py:1754-1803"""
    return _solid_K(_ops.C3D8, coords, elements, E, nu, integral_point, single, device, dtype)


def compute_c3d8_element_stress(coords, elements, displacement, E, nu, integral_point=None, single=True, device="cuda:0",
                                dtype=torch.float32):
    """single=True: ([M,3,3],[M]); single=False: ([M,n_int,3,3],[M,n_int]) (element.py:1696-1752)."""
    return _stress(_ops.C3D8, coords, elements, displacement, E, nu, integral_point, single, device, dtype, False)


def compute_c3d8_M_matrix(coords, elements, rho, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Consistent mass [M,24,24], default 3x3x3 Gauss.  Not in the reference -- parity unpinned."""
    return _solid_M(_ops.C3D8, coords, elements, rho, integral_point, device, dtype)


# ---- C3D20: the reference's implementation (element.py:1852-2188) cannot run -- compute_c3d20_Jacobian raises on an
# einsum subscript mismatch (:1980) and its derivative table is not the serendipity gradient (rows sum to (0.89, 0.88,
# 2.44) at a test point, SURVEY a12).  These functions keep the reference's names and signatures and compute the standard
# 20-node serendipity hex in the node order of the reference's own table and vtk loader (0-7 corners, 8-11 bottom,
# 12-15 top, 16-19 vertical mid-edges).  Parity unpinned; validated by invariants (tests/).

def c3d20_to_c3d4(c3d20_elements, device="cuda:0"):
    """The reference's 24-tet table as written (element.py:1852-1896)."""
    return _ops.to_c3d4(_ops.C3D20, c3d20_elements, device)


def c3d20_integration_points(device="cuda:0", dtype=torch.float32):
    """3x3x3 Gauss, xi slowest, +-sqrt(3/5) rounded to fp32 (q1) (element.py:1898-1919)."""
    return _points_out(_ops.C3D20, device, dtype)


def compute_c3d20_Jacobian(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """[M,3,3] (signature of element.py:1921-1984)."""
    return _solid(_ops.C3D20, 0, coords, elements, integral_point, device, dtype)


def compute_c3d20_shape_gradients(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """[M,20,3] (signature of element.py:1986-2044)."""
    return _solid(_ops.C3D20, 1, coords, elements, integral_point, device, dtype)


def compute_c3d20_B_matrix(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """[M,6,60] (signature of element.py:2046-2074)."""
    return _solid(_ops.C3D20, 2, coords, elements, integral_point, device, dtype)


def compute_c3d20_element_stress(coords, elements, displacement, E, nu, integral_point=None, single=True, device="cuda:0",
                                 dtype=torch.float32):
    """single=True: ([M,3,3],[M]); single=False: ([M,n_int,3,3],[M,n_int]) (signature of element.py:2076-2138)."""
    return _stress(_ops.C3D20, coords, elements, displacement, E, nu, integral_point, single, device, dtype, False)


def compute_c3d20_K_matrix(coords, elements, E, nu, integral_point=None, single=True, device="cuda:0", dtype=torch.float32):
    """[M,60,60]; single=False -> [n_int,M,60,60] unweighted (signature of element.py:2140-2188)."""
    return _solid_K(_ops.C3D20, coords, elements, E, nu, integral_point, single, device, dtype)


def compute_c3d20_M_matrix(coords, elements, rho, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Consistent mass [M,60,60], default 3x3x3 Gauss.  Not in the reference -- parity unpinned."""
    return _solid_M(_ops.C3D20, coords, elements, rho, integral_point, device, dtype)


# ------------------------------------------------------------------------------------------- wedges

def compute_wedge_volumes(coords, elements, device="cuda:0", dtype=torch.float32):
    """element.py:2198-2232"""
    return _ops.volumes(_ops.C3D6, coords, elements, device, dtype)


def compute_wedge_surface_faces_with_extra_node(elements, device="cuda:0"):
    """([quads, tris], [quad_extra, tri_extra]); the two kinds are grouped separately (element.py:2234-2283)."""
    q, qe, _ = _ops.entities(_ops.ENT_WEDGE_QUADS, elements, device, want_shared=False)
    t, te, _ = _ops.entities(_ops.ENT_WEDGE_TRIS, elements, device, want_shared=False)
    return [q, t], [qe, te]


def compute_wedge_surface_normals(coords, elements, device="cuda:0", dtype=torch.float32):
    """element.py:2285-2338 (quads use nodes 0,1,3 of the face; triangles 0,1,2)."""
    (q, t), (qe, te) = compute_wedge_surface_faces_with_extra_node(elements, device)
    return [_ops.surface_normals(coords, q, qe, 3, device, dtype), _ops.surface_normals(coords, t, te, 2, device, dtype)]


def compute_wedge_normals_and_area(coords, elements, device="cuda:0", dtype=torch.float32):
    """[M,5,3] UNIT normals of the faces (0,1,4,3) (1,2,5,4) (2,0,3,5) (0,2,1) (3,4,5), not re-oriented -- despite its name the
    reference neither area-weights nor orients them (element.py:2377-2420)."""
    return _ops.wedge_face_normals(coords, elements, device, dtype)


def c3d6_to_c3d4(element, device="cuda:0"):
    """element.py:2424-2446"""
    return _ops.to_c3d4(_ops.C3D6, element, device)


def c3d6_integration_points(device="cuda:0", dtype=torch.float32):
    """3 triangle points x 2 fp32-rounded line points, weights summing to 2 (element.py:2448-2480)."""
    return _points_out(_ops.C3D6, device, dtype)


def compute_c3d6_Jacobian(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """element.py:2482-2509"""
    return _solid(_ops.C3D6, 0, coords, elements, integral_point, device, dtype)


def compute_c3d6_shape_gradients(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """element.py:2511-2539"""
    return _solid(_ops.C3D6, 1, coords, elements, integral_point, device, dtype)


def compute_c3d6_B_matrix(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    """element.py:2541-2568"""
    return _solid(_ops.C3D6, 2, coords, elements, integral_point, device, dtype)


def compute_c3d6_K_matrix(coords, elements, E, nu, integral_point=None, single=True, device="cuda:0", dtype=torch.float32):
    """single=True (the reference's default) is the one-point centroid rule times the 3-tet |volume|; single=False the
    weighted 6-point rule with signed detJ (element.py:2631-2676)."""
    if single:
        centroid = _pts(_ops.C3D6, torch.tensor([[1 / 3, 1 / 3, 0.0, 1.0]], dtype=torch.float64), dtype)
        return _ops.solid(_ops.C3D6, 5, coords, elements, centroid, E, nu, device, dtype)
    return _solid(_ops.C3D6, 3, coords, elements, integral_point, device, dtype, E, nu, single_point=False)


def compute_c3d6_element_stress(coords, elements, displacement, E, nu, integral_point=None, single=True, device="cuda:0",
                                dtype=torch.float32):
    """single=True: 6-point weighted sums ([M,3,3],[M]); single=False: ([M,n_int,3,3],[M,n_int]) (element.py:2570-2629)."""
    return _stress(_ops.C3D6, coords, elements, displacement, E, nu, integral_point, single, device, dtype, False)


def compute_c3d6_M_matrix(coords, elements, rho, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Consistent mass [M,18,18], default degree-4 triangle rule x 3-point Gauss.  Not in the reference -- parity unpinned."""
    return _solid_M(_ops.C3D6, coords, elements, rho, integral_point, device, dtype)


# ---- C3D15: a header only in the reference (element.py:2679); its dispatchers name compute_c3d15_* functions that do not
# exist (:377-426 -> NameError).  Standard 15-node wedge: 0-2 bottom, 3-5 top corners, 6-8 bottom mid-edges (0,1),(1,2),(2,0),
# 9-11 top mid-edges, 12-14 vertical mid-edges; natural coordinates as C3D6.  Parity unpinned; validated by invariants.

def c3d15_integration_points(device="cuda:0", dtype=torch.float32):
    """9 points: 3-point triangle rule x 3-point Gauss, weights sum to 1 (the wedge's natural volume)."""
    return _points_out(_ops.C3D15, device, dtype)


def compute_c3d15_Jacobian(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    return _solid(_ops.C3D15, 0, coords, elements, integral_point, device, dtype)


def compute_c3d15_shape_gradients(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    return _solid(_ops.C3D15, 1, coords, elements, integral_point, device, dtype)


def compute_c3d15_B_matrix(coords, elements, integral_point, device="cuda:0", dtype=torch.float32):
    return _solid(_ops.C3D15, 2, coords, elements, integral_point, device, dtype)


def compute_c3d15_element_stress(coords, elements, displacement, E, nu, integral_point=None, single=True, device="cuda:0",
                                 dtype=torch.float32):
    return _stress(_ops.C3D15, coords, elements, displacement, E, nu, integral_point, single, device, dtype, False)


def compute_c3d15_K_matrix(coords, elements, E, nu, integral_point=None, single=True, device="cuda:0", dtype=torch.float32):
    """[M,45,45]; single=False -> [n_int,M,45,45] unweighted."""
    return _solid_K(_ops.C3D15, coords, elements, E, nu, integral_point, single, device, dtype)


def compute_c3d15_M_matrix(coords, elements, rho, integral_point=None, device="cuda:0", dtype=torch.float32):
    """Consistent mass [M,45,45].  Not in the reference -- parity unpinned."""
    return _solid_M(_ops.C3D15, coords, elements, rho, integral_point, device, dtype)


# ------------------------------------------------------------------------------------------- face force balance

def compute_c3d4_surface_forces(normal_vectors, stress_tensors, device="cuda:0"):
    """[M,4,3] = element stress [M,3,3] applied to the area-weighted face normals [M,4,3] (element.py:3343-3360)."""
    return _ops.face_forces(normal_vectors, stress_tensors, device)


def compute_c3d4_shared_face_forces_sum(shared_face_indices, element_forces, device="cuda:0"):
    """[S,3] = sum of the two face forces meeting on every shared face (pairs [S,2,2] from identify_tetrahedral_shared_faces;
    zero everywhere at equilibrium) (element.py:3362-3384)."""
    return _ops.shared_face_forces_sum(shared_face_indices, element_forces, device)


# ------------------------------------------------------------------------------------------- mesh input

_VTK_NEN = {"c3d4": 4, "c3d10": 10, "c3d8": 8, "c3d20": 20, "c3d6": 6, "c3d15": 15, "s3": 3, "s6": 6, "s4": 4, "s8": 8}


def vtk_loader_to_torch(file_path, element_type, device="cuda:0", dtype=torch.float32):
    """(points [N,3] in `dtype`, connectivity [M,nen] int64) of a VTK file whose cells are all of `element_type`
    (element.py:39-90).  The reference reads through pyvista and reshapes the flat `mesh.cells` array
    `[nen, ids.., nen, ids..]` to `[-1, nen+1]`; here libfemb200's own host parser produces that array from legacy `.vtk`
    unstructured grids (ASCII or BINARY, classic or 5.x cell layout).  Like the reference's reshape this raises when the flat
    array is not a whole number of `nen+1` rows, and additionally when a row's count is not `nen` (the reference would return
    garbage there).  Files storing 32-bit coordinates go through float32 exactly as pyvista's `mesh.points` does."""
    if element_type not in _VTK_NEN:
        raise ValueError("Invalid element type.")
    dev = _ops.cuda_device(device)
    nen = _VTK_NEN[element_type]
    pts, cells, _types, is_float = _ops.vtk_read(file_path)
    if cells.size % (nen + 1):
        raise ValueError(f"cannot reshape the cell array of size {cells.size} into rows of {nen + 1}")
    rows = cells.reshape(-1, nen + 1)
    if rows.shape[0] and not (rows[:, 0] == nen).all():
        raise ValueError(f"the file holds cells that are not {element_type} ({nen} nodes per cell)")
    p = torch.from_numpy(pts)
    if is_float:
        p = p.to(torch.float32)
    return p.to(device=dev, dtype=dtype), torch.from_numpy(rows[:, 1:].copy()).to(device=dev, dtype=torch.long)


# ------------------------------------------------------------------------------------------- misc topology

def element_to_edge(elements, device="cuda:0"):
    """Unique sorted tet edges [2,E] (element.py:2687-2713) = strictly upper part of the node-level CSR pattern."""
    dev = _ops.cuda_device(device)
    e = _ops.index(elements, dev)[:, :4].contiguous()
    plan = CsrPlan(e, None, dev)
    crow, col = plan.pattern(1)
    rows = torch.repeat_interleave(torch.arange(plan.n_nodes, device=dev), (crow[1:] - crow[:-1]).long())
    keep = col.long() > rows
    return torch.stack([rows[keep], col[keep].long()])


# ------------------------------------------------------------------------------------------- global assembly (additive API)

def assemble_csr(K, elements, N=None, device="cuda:0", plan=None):
    """COO of subdivision.ipynb cell 6 -> coalesced CSR (the reference never coalesces).  Returns a
    torch.sparse_csr_tensor [N*ndof, N*ndof] (int32 indices, fp64 values) whose pattern equals
    torch.sparse_coo_tensor(...).coalesce().to_sparse_csr() of that COO; duplicates are summed in ascending
    element order (deterministic)."""
    dev = _ops.cuda_device(device)
    K = torch.as_tensor(K)
    nen = elements.shape[1]
    ndof = K.shape[1] // nen
    if plan is None:
        plan = _ops.cached_plan(elements, N if N is not None else int(torch.as_tensor(elements).max().item()) + 1, dev)
    crow, col = plan.pattern(ndof)
    vals = plan.assemble(K, ndof)
    n = plan.n_nodes * ndof
    return torch.sparse_csr_tensor(crow, col, vals, size=(n, n), device=dev)
