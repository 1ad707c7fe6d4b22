"""Thin torch <-> C-ABI plumbing: allocate outputs with torch, pass raw device pointers to libfemb200.

PyTorch is used for device memory and streams only.  Every function requires a CUDA device; a CPU
device raises (the reference's `device="cpu"` path is deliberately not provided: no CPU fallback).
"""
from __future__ import annotations

import collections
import ctypes as C
import os
import weakref

import torch

from . import _lib
from ._lib import CGResult, check, lib

C3D4, C3D6, C3D8, C3D10, C3D15, C3D20, S3, S4 = 4, 6, 8, 10, 15, 20, 103, 104
ENT_TET_FACES, ENT_HEX_FACES, ENT_WEDGE_QUADS, ENT_WEDGE_TRIS, ENT_TRI_EDGES, ENT_QUAD_EDGES = range(6)
_ENT = {ENT_TET_FACES: (4, 3), ENT_HEX_FACES: (6, 4), ENT_WEDGE_QUADS: (3, 4), ENT_WEDGE_TRIS: (2, 3), ENT_TRI_EDGES: (3, 2),
        ENT_QUAD_EDGES: (4, 2)}


def cuda_device(device) -> torch.device:
    d = torch.device(device)
    if d.type != "cuda":
        raise RuntimeError(f"femb200 runs on CUDA devices only (got device={device!r}); there is no CPU fallback")
    if not torch.cuda.is_available():
        raise RuntimeError("femb200 needs a CUDA device (sm_100a); none is visible")
    return d


def _stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def real(t, dev, dtype) -> torch.Tensor:
    if dtype not in (torch.float32, torch.float64):
        raise TypeError(f"dtype must be float32 or float64, got {dtype}")
    return torch.as_tensor(t).to(device=dev, dtype=dtype).contiguous()


def index(t, dev) -> torch.Tensor:
    t = torch.as_tensor(t).to(device=dev)
    if t.dtype not in (torch.int32, torch.int64):
        t = t.to(torch.int64)
    return t.contiguous()


def _fp(t):
    return t.element_size()


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _host_doubles(values):
    arr = (C.c_double * len(values))(*[float(v) for v in values])
    return arr


def default_points(kind) -> list:
    buf = (C.c_double * (64 * 4))()
    n = lib.femb_default_points(kind, buf)
    if n < 0:
        check(1, "femb_default_points")
    return [[buf[4 * q + k] for k in range(4)] for q in range(n)]


def mass_points(kind) -> list:
    buf = (C.c_double * (64 * 4))()
    n = lib.femb_mass_points(kind, buf)
    if n < 0:
        check(1, "femb_mass_points")
    return [[buf[4 * q + k] for k in range(4)] for q in range(n)]


# ----------------------------------------------------------------------------- element kernels

def _out_buffer(out, shape, dev, dtype):
    """`out=` (additive to the reference API): reuse a caller-owned result buffer instead of allocating a new one per call --
    at 64 M tets a [M,4,4] fp64 result is 8.2 GB, and a fresh cudaMalloc of that size costs 15x the kernel."""
    if out is None:
        return torch.empty(shape, device=dev, dtype=dtype)
    if tuple(out.shape) != tuple(shape) or out.dtype != dtype or out.device != torch.device(dev) or not out.is_contiguous():
        raise ValueError(f"out= must be a contiguous {dtype} tensor of shape {tuple(shape)} on {dev}")
    return out


def c3d4(what, coords, elements, E=0.0, nu=0.0, device="cuda:0", dtype=torch.float32, out=None):
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    M = conn.shape[0]
    shape = {0: (M, 4, 3), 1: (M, 6, 12), 2: (M, 12, 12), 3: (M, 4, 4), 4: (M, 12, 12), 5: (M,)}[what]
    out = _out_buffer(out, shape, dev, dtype)
    flag = torch.zeros(1, device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        check(lib.femb_c3d4(what, _p(x), _fp(x), _p(conn), _fp(conn), M, float(E), float(nu), _p(out), _p(flag), _stream(dev)), "femb_c3d4")
    if what in (0, 1, 2, 3) and M and int(flag.item()):   # the reference also synchronises here (torch.any, element.py:857)
        raise ValueError("Singular matrix encountered while computing B matrix.")
    return out


def volumes(kind, coords, elements, device="cuda:0", dtype=torch.float32):
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    M = conn.shape[0]
    out = torch.empty((M,), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        check(lib.femb_elem_volumes(kind, _p(x), _fp(x), _p(conn), _fp(conn), M, conn.shape[1], _p(out), _stream(dev)), "femb_elem_volumes")
    return out


_NEN = {C3D4: 4, C3D6: 6, C3D8: 8, C3D10: 10, C3D15: 15, C3D20: 20, S3: 3, S4: 4}


def solid(kind, what, coords, elements, points, E=0.0, nu=0.0, device="cuda:0", dtype=torch.float32, out=None):
    """points: list of [xi,eta,zeta,w] rows (host)."""
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    nen = _NEN[kind]
    if conn.shape[1] != nen:
        conn = conn[:, :nen].contiguous()
    M, nd, nq = conn.shape[0], 3 * nen, len(points)
    shape = {0: (M, 3, 3), 1: (M, nen, 3), 2: (M, 6, nd), 3: (M, nd, nd), 4: (nq, M, nd, nd), 5: (M, nd, nd), 6: (M, nd, nd)}[what]
    out = _out_buffer(out, shape, dev, dtype)
    flat = [v for row in points for v in row]
    with torch.cuda.device(dev):
        check(lib.femb_solid(kind, what, _p(x), _fp(x), _p(conn), _fp(conn), M, _host_doubles(flat), nq, float(E), float(nu), _p(out),
                             _stream(dev)), "femb_solid")
    return out


def solid_stress(kind, coords, elements, displacement, points, E, nu, single=True, device="cuda:0", dtype=torch.float32):
    """(stress, vm): single -> [M,3,3],[M]; else point-major [nq,M,3,3],[nq,M]."""
    dev = cuda_device(device)
    x, conn, u = real(coords, dev, dtype), index(elements, dev), real(displacement, dev, dtype)
    nen = _NEN[kind]
    if conn.shape[1] != nen:
        conn = conn[:, :nen].contiguous()
    if u.shape != x.shape:
        raise ValueError(f"displacement must be [N,3] like coords, got {tuple(u.shape)} vs {tuple(x.shape)}")
    M, nq = conn.shape[0], len(points)
    lead = (M,) if single else (nq, M)
    S = torch.empty(lead + (3, 3), device=dev, dtype=dtype)
    V = torch.empty(lead, device=dev, dtype=dtype)
    flat = [v for row in points for v in row]
    with torch.cuda.device(dev):
        check(lib.femb_solid_stress(kind, _p(x), _fp(x), _p(conn), _fp(conn), M, _p(u), _host_doubles(flat), nq, float(E), float(nu),
                                    1 if single else 0, _p(S), _p(V), _stream(dev)), "femb_solid_stress")
    return S, V


def stress_helper(what, t):
    """what 0: Voigt [M,6] -> [M,3,3]; 1: [M,3,3] -> von Mises [M].  Works on the tensor's own device/dtype like the reference."""
    t = torch.as_tensor(t)
    dev = cuda_device(t.device)
    t = real(t, dev, t.dtype)
    M = t.shape[0]
    out = torch.empty((M, 3, 3) if what == 0 else (M,), device=dev, dtype=t.dtype)
    with torch.cuda.device(dev):
        check(lib.femb_stress_helper(what, _p(t), _fp(t), M, _p(out), _stream(dev)), "femb_stress_helper")
    return out


def shell(kind, what, coords, elements, points=None, D=None, device="cuda:0", dtype=torch.float32):
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    nen = _NEN[kind]
    M, nd = conn.shape[0], 6 * nen
    points = points if points is not None else [[0.0, 0.0, 0.0, 1.0]]
    nq = len(points)
    shape = {0: (M, 3, 3), 1: (M, 2, 2), 2: (M, nen, 2), 3: (M, 6, nd), 4: (M, nd, nd), 5: (M, nd, nd, nq)}[what]
    out = torch.empty(shape, device=dev, dtype=dtype)
    flat = [v for row in points for v in row]
    Dh = _host_doubles([float(v) for v in D.reshape(-1).tolist()]) if D is not None else None
    with torch.cuda.device(dev):
        check(lib.femb_shell(kind, what, _p(x), _fp(x), _p(conn), _fp(conn), M, _host_doubles(flat), nq, Dh, _p(out), _stream(dev)),
              "femb_shell")
    return out


def shell_ex(kind, what, coords, elements, factors=None, D=None, disp=None, device="cuda:0", dtype=torch.float32):
    """femb_shell_ex: factors = [[1-xi, 1+xi, 1-eta, 1+eta, w], ...] (host; S3 ignores them).  what 7: sum_q w_q B_q [M,6,nd]; 8: per-point [M,6,nd,nq]; 9: stress resultants [M,6] from disp [N,6]."""
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    nen = _NEN[kind]
    M, nd = conn.shape[0], 6 * nen
    factors = factors if factors is not None else [[1.0, 1.0, 1.0, 1.0, 1.0]]
    nq = len(factors)
    shape = {0: (M, 3, 3), 1: (M, 2, 2), 2: (M, nen, 2), 3: (M, 6, nd), 4: (M, nd, nd), 5: (M, nd, nd, nq), 7: (M, 6, nd),
             8: (M, 6, nd, nq), 9: (M, 6)}[what]
    out = torch.empty(shape, device=dev, dtype=dtype)
    u = real(disp, dev, dtype) if disp is not None else None
    if what == 9 and (u is None or u.dim() != 2 or u.shape[1] != 6 or u.shape[0] != x.shape[0]):
        raise ValueError("shell stress needs the displacement as [N,6] (one row per node of coords)")
    flat = [v for row in factors for v in row]
    Dh = _host_doubles([float(v) for v in D.reshape(-1).tolist()]) if D is not None else None
    with torch.cuda.device(dev):
        check(lib.femb_shell_ex(kind, what, _p(x), _fp(x), _p(conn), _fp(conn), M, _host_doubles(flat), nq, Dh, _p(u), _p(out), _stream(dev)),
              "femb_shell_ex")
    return out


def shell_normal(coords, elements, device="cuda:0"):
    """[M,3]: S3 cross(x1-x0, x2-x0)/2, S4 cross(x1-x0, x3-x0), in the dtype of `coords`."""
    dev = cuda_device(device)
    x = torch.as_tensor(coords)
    x = real(x, dev, x.dtype if x.dtype in (torch.float32, torch.float64) else torch.float32)
    conn = index(elements, dev)
    out = torch.empty((conn.shape[0], 3), device=dev, dtype=x.dtype)
    with torch.cuda.device(dev):
        check(lib.femb_shell_normal(_p(x), _fp(x), _p(conn), _fp(conn), conn.shape[0], conn.shape[1], _p(out), _stream(dev)), "femb_shell_normal")
    return out


def shell_rotate_K(K, unit):
    """[M,nd,nd] = T^T K T with T = blockdiag(unit, ...): the shell element operator in global axes (fp64)."""
    dev = K.device
    K = real(K, dev, torch.float64)
    R = real(unit, dev, torch.float64)
    M, nd, _ = K.shape
    if tuple(R.shape) != (M, 3, 3):
        raise ValueError(f"unit must be [M,3,3], got {tuple(R.shape)}")
    out = torch.empty_like(K)
    with torch.cuda.device(dev):
        check(lib.femb_shell_rotate_operator(_p(K), _p(R), 8, M, nd, _p(out), _stream(dev)), "femb_shell_rotate_operator")
    return out


def shell_local_coordinates(coords, elements, unit, device="cuda:0", dtype=torch.float32):
    """[M,nen,3]: node coordinates relative to node 0 of each element, expressed in the frame `unit` [M,3,3]."""
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    R = real(unit, dev, dtype)
    M, nen = conn.shape
    if tuple(R.shape) != (M, 3, 3):
        raise ValueError(f"unit must be [M,3,3], got {tuple(R.shape)}")
    out = torch.empty((M, nen, 3), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        check(lib.femb_shell_local_coordinates(_p(x), _fp(x), _p(conn), _fp(conn), M, nen, _p(R), _p(out), _stream(dev)),
              "femb_shell_local_coordinates")
    return out


def shell_local_displacement(elements, displacement, unit, device="cuda:0"):
    """[M,nen,6]: nodal translations and rotations of every element in its own frame (dtype of `displacement`)."""
    dev = cuda_device(device)
    conn = index(elements, dev)
    u = torch.as_tensor(displacement)
    u = real(u, dev, u.dtype if u.dtype in (torch.float32, torch.float64) else torch.float32)
    R = real(unit, dev, u.dtype)
    M, nen = conn.shape
    if u.dim() != 2 or u.shape[1] != 6 or tuple(R.shape) != (M, 3, 3):
        raise ValueError(f"expected displacement [N,6] and unit [M,3,3], got {tuple(u.shape)} and {tuple(R.shape)}")
    out = torch.empty((M, nen, 6), device=dev, dtype=u.dtype)
    with torch.cuda.device(dev):
        check(lib.femb_shell_local_displacement(_p(conn), _fp(conn), M, nen, _p(u), _p(R), _fp(u), _p(out), _stream(dev)),
              "femb_shell_local_displacement")
    return out


def shell_postprocess(NMQ, t, z, device="cuda:0", dtype=torch.float32):
    """[8,M]: sx, sy, txy, s1, s2, theta_p, tau_max, vm."""
    dev = cuda_device(device)
    v = real(NMQ, dev, dtype)
    if v.dim() != 2 or v.shape[1] < 6:
        raise ValueError(f"NMQ must be [M,6] or [M,8], got {tuple(v.shape)}")
    M = v.shape[0]
    out = torch.empty((8, M), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        check(lib.femb_shell_postprocess(_p(v), _fp(v), M, v.shape[1], float(t), float(z), _p(out), _stream(dev)), "femb_shell_postprocess")
    return out


def face_forces(normals, stress, device="cuda:0"):
    dev = cuda_device(device)
    s = torch.as_tensor(stress)
    dt = s.dtype if s.dtype in (torch.float32, torch.float64) else torch.float32
    s, n = real(s, dev, dt), real(normals, dev, dt)
    M, nf = n.shape[0], n.shape[1]
    if tuple(s.shape) != (M, 3, 3) or n.shape[2] != 3:
        raise ValueError(f"expected normals [M,nf,3] and stress [M,3,3], got {tuple(n.shape)} and {tuple(s.shape)}")
    out = torch.empty((M, nf, 3), device=dev, dtype=dt)
    with torch.cuda.device(dev):
        check(lib.femb_face_forces(_p(n), _p(s), _fp(s), M, nf, _p(out), _stream(dev)), "femb_face_forces")
    return out


def shared_face_forces_sum(pairs, forces, device="cuda:0"):
    dev = cuda_device(device)
    pr = torch.as_tensor(pairs).to(device=dev, dtype=torch.int64).contiguous()
    f = torch.as_tensor(forces)
    f = real(f, dev, f.dtype if f.dtype in (torch.float32, torch.float64) else torch.float32)
    S = pr.shape[0]
    if tuple(pr.shape[1:]) != (2, 2) or f.dim() != 3 or f.shape[2] != 3:
        raise ValueError(f"expected pairs [S,2,2] and forces [M,nf,3], got {tuple(pr.shape)} and {tuple(f.shape)}")
    if S and (int(pr[:, :, 0].max()) >= f.shape[0] or int(pr[:, :, 1].max()) >= f.shape[1] or int(pr.min()) < 0):
        raise IndexError("shared-face pair refers to an element / local face outside element_forces")
    out = torch.empty((S, 3), device=dev, dtype=f.dtype)
    with torch.cuda.device(dev):
        check(lib.femb_shared_face_forces_sum(_p(pr), S, _p(f), _fp(f), f.shape[1], _p(out), _stream(dev)), "femb_shared_face_forces_sum")
    return out


def wedge_face_normals(coords, elements, device="cuda:0", dtype=torch.float32):
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    out = torch.empty((conn.shape[0], 5, 3), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        check(lib.femb_wedge_face_normals(_p(x), _fp(x), _p(conn), _fp(conn), conn.shape[0], conn.shape[1], _p(out), _stream(dev)),
              "femb_wedge_face_normals")
    return out


def shell_extrude(coords, tri, quad, thickness, eps=1e-8, device="cuda:0", dtype=torch.float32):
    """(coords3d [2N,3], wedges [T,6], hexahedra [S,8]) from a mid-surface mesh; connectivity keeps its integer dtype."""
    dev = cuda_device(device)
    x = real(coords, dev, dtype)
    N = x.shape[0]
    conns, plans, outs = [], [], []
    for c, nen in ((tri, 3), (quad, 4)):
        c = index(c if c is not None else torch.empty((0, nen), dtype=torch.int64), dev).reshape(-1, nen)
        if c.numel() and (int(c.max()) >= N or int(c.min()) < 0):
            raise IndexError("shell connectivity refers to a node outside coords")
        conns.append(c)
        plans.append(cached_plan(c, N, dev) if c.shape[0] else None)
        outs.append(torch.empty((c.shape[0], 2 * nen), device=dev, dtype=c.dtype))
    x3 = torch.empty((2 * N, 3), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        st = _stream(dev)
        check(lib.femb_shell_extrude(plans[0].handle if plans[0] else None, plans[1].handle if plans[1] else None, _p(x), _fp(x), N,
                                     float(thickness), float(eps), _p(x3), st), "femb_shell_extrude")
        for c, o, nen in zip(conns, outs, (3, 4)):
            check(lib.femb_extrude_connectivity(_p(c), _fp(c), c.shape[0], nen, N, _p(o), st), "femb_extrude_connectivity")
    return x3, outs[0], outs[1]


def vtk_read(file_path):
    """Host parse of a legacy .vtk unstructured grid -> (points float64 [n,3] (numpy), flat cells int64 (pyvista's mesh.cells
    layout), cell types int32 or None, points_are_float)."""
    import numpy as np
    h, npnt, ncell, csize, isf = C.c_void_p(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int32()
    check(lib.femb_vtk_open(str(file_path).encode(), C.byref(h), C.byref(npnt), C.byref(ncell), C.byref(csize), C.byref(isf)), "femb_vtk_open")
    try:
        pts = np.empty((npnt.value, 3), dtype=np.float64)
        cells = np.empty(csize.value, dtype=np.int64)
        types = np.empty(ncell.value, dtype=np.int32)
        check(lib.femb_vtk_read(h, pts.ctypes.data_as(C.c_void_p), cells.ctypes.data_as(C.c_void_p), None), "femb_vtk_read")
        if lib.femb_vtk_read(h, None, None, types.ctypes.data_as(C.c_void_p)) != 0:
            types = None
    finally:
        lib.femb_vtk_close(h)
    return pts, cells, types, bool(isf.value)


def to_c3d4(kind, elements, device="cuda:0"):
    dev = cuda_device(device)
    conn = index(elements, dev)
    k = {C3D10: 8, C3D8: 6, C3D6: 3, C3D20: 24}[kind]
    if conn.shape[1] != _NEN[kind]:
        conn = conn[:, :_NEN[kind]].contiguous()
    out = torch.empty((conn.shape[0] * k, 4), device=dev, dtype=torch.int64)
    with torch.cuda.device(dev):
        check(lib.femb_to_c3d4(kind, _p(conn), _fp(conn), conn.shape[0], _p(out), _stream(dev)), "femb_to_c3d4")
    return out


# ----------------------------------------------------------------------------- topology

def entities(ent_kind, elements, device="cuda:0", want_surface=True, want_shared=True):
    """Returns (faces [K,nfn], extra [K], pairs [S,2,2]) -- entries not requested are None."""
    dev = cuda_device(device)
    conn = index(elements, dev)
    M = conn.shape[0]
    nf, nfn = _ENT[ent_kind]
    plan, K, S = C.c_void_p(), C.c_int64(), C.c_int64()
    with torch.cuda.device(dev):
        st = _stream(dev)
        check(lib.femb_entities_create(ent_kind, _p(conn), _fp(conn), M, conn.shape[1], st, C.byref(plan), C.byref(K), C.byref(S)),
              "femb_entities_create")
        try:
            faces = extra = pairs = None
            if want_surface:
                faces = torch.empty((K.value, nfn), device=dev, dtype=torch.int64)
                extra = torch.empty((K.value,), device=dev, dtype=torch.int64)
                check(lib.femb_entities_surface(plan, _p(faces), _p(extra), st), "femb_entities_surface")
            if want_shared:
                pairs = torch.empty((S.value, 2, 2), device=dev, dtype=torch.int64)
                check(lib.femb_entities_shared(plan, _p(pairs), st), "femb_entities_shared")
            torch.cuda.current_stream(dev).synchronize()   # plan scratch is freed below
        finally:
            lib.femb_entities_destroy(plan)
    return faces, extra, pairs


def surface_normals(coords, faces, extra, second, device="cuda:0", dtype=torch.float32):
    dev = cuda_device(device)
    x = real(coords, dev, dtype)
    out = torch.empty((faces.shape[0], 3), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        check(lib.femb_surface_normals(_p(x), _fp(x), _p(faces), _p(extra), faces.shape[0], faces.shape[1], second, _p(out), _stream(dev)),
              "femb_surface_normals")
    return out


def face_normals_area(kind, coords, elements, device="cuda:0", dtype=torch.float32):
    dev = cuda_device(device)
    x, conn = real(coords, dev, dtype), index(elements, dev)
    nf = 4 if kind == C3D4 else 6
    out = torch.empty((conn.shape[0], nf, 3), device=dev, dtype=dtype)
    with torch.cuda.device(dev):
        check(lib.femb_face_normals_area(kind, _p(x), _fp(x), _p(conn), _fp(conn), conn.shape[0], conn.shape[1], _p(out), _stream(dev)),
              "femb_face_normals_area")
    return out


# ----------------------------------------------------------------------------- assembly plan

class CsrPlan:
    """Node-level sparsity pattern + node->element incidence of one connectivity array (device resident)."""

    def __init__(self, elements, n_nodes=None, device="cuda:0"):
        self.dev = cuda_device(device)
        conn = index(elements, self.dev)
        self.M, self.nen = conn.shape
        self.n_nodes = int(n_nodes) if n_nodes is not None else (int(conn.max().item()) + 1 if self.M else 1)
        h, nnz = C.c_void_p(), C.c_int64()
        with torch.cuda.device(self.dev):
            try:
                check(lib.femb_csr_plan_create(_p(conn), _fp(conn), self.M, self.nen, self.n_nodes, _stream(self.dev), C.byref(h), C.byref(nnz)),
                      "femb_csr_plan_create")
            except _lib.FembError as exc:
                if "outside [0, n_nodes)" in str(exc):   # the reference's gathers raise an index error for such connectivity
                    raise IndexError(f"connectivity holds a node index outside [0, {self.n_nodes})") from exc
                raise
        self.handle, self.nnz_nodes = h, nnz.value
        # device bytes held by the plan (conn32, incidences, slot table, pattern, P1 records once built): bounds the plan cache
        L = self.M * self.nen
        self.nbytes = L * (8 + self.nen) + 8 * (self.n_nodes + 1) + 4 * self.nnz_nodes + (20 * L if self.nen == 4 else 0)
        self._fin = weakref.finalize(self, lib.femb_csr_plan_destroy, h)
        self._patterns = {}

    def pattern(self, ndof):
        """(crow int32 [n+1], col int32 [nnz]) for `ndof` dofs per node."""
        if ndof not in self._patterns:
            n = self.n_nodes * ndof
            crow = torch.empty(n + 1, device=self.dev, dtype=torch.int32)
            col = torch.empty(self.nnz_nodes * ndof * ndof, device=self.dev, dtype=torch.int32)
            with torch.cuda.device(self.dev):
                check(lib.femb_csr_plan_pattern(self.handle, ndof, _p(crow), _p(col), _stream(self.dev)), "femb_csr_plan_pattern")
            self._patterns[ndof] = (crow, col)
        return self._patterns[ndof]

    def assemble(self, Ke, ndof, out=None):
        """CSR values (fp64) from materialised element matrices Ke [M, nen*ndof, nen*ndof]."""
        Ke = real(Ke, self.dev, torch.float64)
        assert Ke.shape == (self.M, self.nen * ndof, self.nen * ndof), (Ke.shape, self.M, self.nen, ndof)
        vals = out if out is not None else torch.empty(self.nnz_nodes * ndof * ndof, device=self.dev, dtype=torch.float64)
        with torch.cuda.device(self.dev):
            check(lib.femb_csr_assemble(self.handle, ndof, _p(Ke), _p(vals), _stream(self.dev)), "femb_csr_assemble")
        return vals

    def assemble_c3d4(self, coords, kind, E=0.0, nu=0.0, out=None, check_singular=True):
        """Fused P1-tet assembly from coordinates. kind: 'poisson' (1 dof) or 'elasticity' (3 dofs)."""
        k = {"poisson": 0, "elasticity": 1}[kind]
        d2 = 1 if k == 0 else 9
        x = real(coords, self.dev, torch.float64)
        vals = out if out is not None else torch.empty(self.nnz_nodes * d2, device=self.dev, dtype=torch.float64)
        flag = torch.zeros(1, device=self.dev, dtype=torch.int32)
        with torch.cuda.device(self.dev):
            check(lib.femb_csr_assemble_c3d4(self.handle, k, _p(x), float(E), float(nu), _p(vals), _p(flag), _stream(self.dev)),
                  "femb_csr_assemble_c3d4")
        if check_singular and int(flag.item()):
            raise ValueError("Singular matrix encountered while computing B matrix.")
        return vals

    def ebe_apply(self, Ke, u, ndof, unit=None, dtype=torch.float64):
        Ke, u = real(Ke, self.dev, dtype), real(u, self.dev, dtype)
        un = real(unit, self.dev, dtype) if unit is not None else None
        y = torch.empty((self.n_nodes, ndof), device=self.dev, dtype=dtype)
        assert u.shape[0] == self.n_nodes, "displacement rows must equal the plan's node count"
        with torch.cuda.device(self.dev):
            check(lib.femb_ebe_apply(self.handle, ndof, _p(Ke), _p(u), _p(un), _fp(u), _p(y), _stream(self.dev)), "femb_ebe_apply")
        return y

    def ebe_diag(self, Ke, ndof, dtype=torch.float64, col0=False):
        """[N, ndof] diagonal of sum_e K_e (element-ascending sums); col0=True sums column 0 of every row instead."""
        Ke = real(Ke, self.dev, dtype)
        assert Ke.shape == (self.M, self.nen * ndof, self.nen * ndof), (Ke.shape, self.M, self.nen, ndof)
        out = torch.empty((self.n_nodes, ndof), device=self.dev, dtype=dtype)
        with torch.cuda.device(self.dev):
            check(lib.femb_ebe_diag(self.handle, ndof, _p(Ke), _fp(Ke), 1 if col0 else 0, _p(out), _stream(self.dev)), "femb_ebe_diag")
        return out

    def node_average(self, elem_values, dtype=None):
        """[N] mean over the elements containing each node (0 for isolated nodes), ascending element order."""
        v = torch.as_tensor(elem_values)
        v = real(v, self.dev, dtype if dtype is not None else (v.dtype if v.dtype in (torch.float32, torch.float64) else torch.float64))
        assert v.shape == (self.M,), (v.shape, self.M)
        out = torch.empty(self.n_nodes, device=self.dev, dtype=v.dtype)
        with torch.cuda.device(self.dev):
            check(lib.femb_node_average(self.handle, _p(v), _fp(v), _p(out), _stream(self.dev)), "femb_node_average")
        return out


def p1_to_p2(coords, elements, device, dtype):
    """Mid-edge insertion on the device (csrc/refine.cu): (coords' [N+E,3] dtype, conn10 [M,10] int32, edges [E,2] int32 = end
    points of new node N+r).  Numbering = the reference's first-encounter order (element.py:777-833)."""
    dev = cuda_device(device)
    x = torch.as_tensor(coords).to(dev)
    if x.dtype not in (torch.float32, torch.float64):
        x = x.to(torch.float64)
    x = x.contiguous()
    conn = index(elements, dev)
    M, N = conn.shape[0], x.shape[0]
    h, ne = C.c_void_p(), C.c_int64()
    with torch.cuda.device(dev):
        check(lib.femb_p2_create(_p(conn), _fp(conn), M, N, _stream(dev), C.byref(h), C.byref(ne)), "femb_p2_create")
        try:
            E = ne.value
            conn10 = torch.empty((M, 10), device=dev, dtype=torch.int32)
            xo = torch.empty((N + E, 3), device=dev, dtype=dtype)
            edges = torch.empty((E, 2), device=dev, dtype=torch.int32)
            check(lib.femb_p2_fill(h, _p(conn), _fp(conn), _p(x), _fp(x), xo.element_size(), _p(conn10), _p(xo), _p(edges), _stream(dev)),
                  "femb_p2_fill")
        finally:
            lib.femb_p2_destroy(h)
    return xo, conn10, edges


_PLAN_CACHE: "collections.OrderedDict" = collections.OrderedDict()
PLAN_CACHE_BYTES = int(float(os.environ.get("FEMB_PLAN_CACHE_GB", "16")) * 2 ** 30)   # a 64 M-tet plan holds ~8 GB of HBM


def cached_plan(elements, n_nodes, device) -> CsrPlan:
    """Plans are cached per connectivity TENSOR (object identity + in-place version counter) so that repeated operator
    applications on the same mesh (every CG iteration of the reference calls compute_nodal_forces) reuse one plan.
    Only torch tensors handed in by the caller are cached: numpy arrays / lists have no version counter, so an in-place
    renumbering would silently reuse a stale plan -- they get a fresh plan per call.  The cache is bounded by the device
    bytes the plans hold (FEMB_PLAN_CACHE_GB, default 16), least recently used first, and by 8 entries."""
    if not torch.is_tensor(elements):
        return CsrPlan(torch.as_tensor(elements).clone(), n_nodes, device)
    e = elements
    key = (id(e), e.data_ptr(), tuple(e.shape), e.dtype, e._version, str(e.device), int(n_nodes), str(device))
    plan = _PLAN_CACHE.get(key)
    if plan is None:
        plan = CsrPlan(e, n_nodes, device)
        plan._keepalive = e   # keeps id() / data_ptr from being recycled while cached
        _PLAN_CACHE[key] = plan
        while len(_PLAN_CACHE) > 1 and (len(_PLAN_CACHE) > 8 or sum(p.nbytes for p in _PLAN_CACHE.values()) > PLAN_CACHE_BYTES):
            _PLAN_CACHE.popitem(last=False)
    else:
        _PLAN_CACHE.move_to_end(key)
    return plan


# ----------------------------------------------------------------------------- Krylov

def spmv(crow, col, val, x):
    dev = val.device
    n = crow.numel() - 1
    xx = x.reshape(-1).contiguous()
    y = torch.empty(n, device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        check(lib.femb_spmv(n, val.numel(), _p(crow), _p(col), _p(val), _p(xx), _p(y), _stream(dev)), "femb_spmv")
    return y.reshape(x.shape) if x.numel() == n else y          # rectangular operators (restriction) return [n]


def jacobi(crow, col, val, mask=None):
    dev = val.device
    n = crow.numel() - 1
    out = torch.empty(n, device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        check(lib.femb_csr_jacobi(n, _p(crow), _p(col), _p(val), _p(mask), _p(out), _stream(dev)), "femb_csr_jacobi")
    return out


STATUS = {0: "converged", 1: "breakdown", 2: "maxiter"}


def cg_solve(crow, col, val, F, mask=None, minv=None, u_init=None, tol=1e-10, max_iter=1000, eps=1e-30, check_every=16):
    """Runs the reference CG (mask: uint8 per dof, 0 = held at zero) or PCG (minv given) loop on the device.
    Returns (u [same shape as F], info dict)."""
    dev = val.device
    n = crow.numel() - 1
    Ff = F.to(device=dev, dtype=torch.float64).reshape(-1).contiguous()
    assert Ff.numel() == n, (Ff.numel(), n)
    u = torch.zeros(n, device=dev, dtype=torch.float64) if u_init is None else \
        u_init.to(device=dev, dtype=torch.float64).reshape(-1).clone().contiguous()
    work = torch.empty(4 * n, device=dev, dtype=torch.float64)
    res = CGResult()
    with torch.cuda.device(dev):
        check(lib.femb_cg_solve(n, val.numel(), _p(crow), _p(col), _p(val), _p(Ff), _p(mask), _p(minv), _p(u), _p(work), float(tol),
                                int(max_iter), float(eps), int(check_every), C.byref(res), _stream(dev)), "femb_cg_solve")
    info = {"iterations": res.iterations, "status": STATUS.get(res.status, "?"), "rs": res.rs, "loop_ms": res.loop_ms,
            "index_bytes": res.index_bytes}
    return u.reshape(F.shape), info


def cg_solve_multi(mats, F, mask=None, minv=None, u_init=None, tol=1e-10, max_iter=1000, eps=1e-30, check_every=16):
    """cg_solve with the operator given as a sum of CSR triples [(crow, col, val), ...] over the same rows."""
    dev = mats[0][2].device
    n = mats[0][0].numel() - 1
    Ff = F.to(device=dev, dtype=torch.float64).reshape(-1).contiguous()
    assert Ff.numel() == n and all(m[0].numel() - 1 == n for m in mats)
    u = torch.zeros(n, device=dev, dtype=torch.float64) if u_init is None else \
        u_init.to(device=dev, dtype=torch.float64).reshape(-1).clone().contiguous()
    work = torch.empty(4 * n, device=dev, dtype=torch.float64)
    k = len(mats)
    nnz = (C.c_int64 * k)(*[m[2].numel() for m in mats])
    crow = (C.c_void_p * k)(*[m[0].data_ptr() for m in mats])
    col = (C.c_void_p * k)(*[m[1].data_ptr() for m in mats])
    val = (C.c_void_p * k)(*[m[2].data_ptr() for m in mats])
    res = CGResult()
    with torch.cuda.device(dev):
        check(lib.femb_cg_solve_multi(n, k, nnz, crow, col, val, _p(Ff), _p(mask), _p(minv), _p(u), _p(work), float(tol), int(max_iter),
                                      float(eps), int(check_every), C.byref(res), _stream(dev)), "femb_cg_solve_multi")
    info = {"iterations": res.iterations, "status": STATUS.get(res.status, "?"), "rs": res.rs, "loop_ms": res.loop_ms}
    return u.reshape(F.shape), info


def cg_solve_operator(apply, R, tol=1e-8, max_iter=1000, check_every=8, device="cuda:0"):
    """CG on y = apply(x) (torch fp64 vectors of R's shape in, same shape out) -- the reference's conjugate_gradient_solver_Ku loop.
    The library drives the loop and calls back for the operator; exceptions raised by `apply` are re-raised here."""
    dev = cuda_device(device)
    Rf = R.to(device=dev, dtype=torch.float64).reshape(-1).contiguous()
    n = Rf.numel()
    u = torch.zeros(n, device=dev, dtype=torch.float64)
    work = torch.empty(3 * n, device=dev, dtype=torch.float64)
    views = {u.data_ptr(): u, (work.data_ptr() + 8 * n): work[n:2 * n]}   # the two vectors the loop ever applies the operator to
    Ap = work[2 * n:]
    raised = []

    def _cb(_ctx, xptr, yptr, _stream_):
        try:
            x = views[int(xptr)]
            assert int(yptr) == Ap.data_ptr()
            y = apply(x.reshape(R.shape))
            Ap.copy_(torch.as_tensor(y).to(device=dev, dtype=torch.float64).reshape(-1))
            return 0
        except BaseException as exc:   # noqa: BLE001  (must not propagate through the C frame)
            raised.append(exc)
            return 1

    cb = _lib.APPLY_FN(_cb)
    res = CGResult()
    with torch.cuda.device(dev):
        rc = lib.femb_cg_solve_operator(n, cb, None, _p(Rf), _p(u), _p(work), float(tol), int(max_iter), int(check_every), C.byref(res),
                                        _stream(dev))
    if raised:
        raise raised[0]
    check(rc, "femb_cg_solve_operator")
    info = {"iterations": res.iterations, "status": STATUS.get(res.status, "?"), "rs": res.rs, "loop_ms": res.loop_ms}
    return u.reshape(R.shape), info


# ----------------------------------------------------------------------------- tall-skinny vectors (modal solver)

class MultiVec:
    """k vectors of length n stored one after the other (fp64): `data` is [k, n] contiguous, column j = data[j]."""

    def __init__(self, data):
        assert data.dim() == 2 and data.dtype == torch.float64 and data.is_contiguous() and data.shape[0] <= 8
        self.data, self.k, self.n, self.dev = data, data.shape[0], data.shape[1], data.device

    @classmethod
    def from_columns(cls, X, dev):
        """From the reference's layout [n, k] (any float dtype)."""
        return cls(torch.as_tensor(X).to(device=dev, dtype=torch.float64).t().contiguous())

    def columns(self):
        return self.data.t().contiguous()

    def cols(self, a, b):
        return MultiVec(self.data[a:b])

    def gram(self, other, w=None):
        """[k_self, k_other] host tensor: sum_r self_i[r] w[r] other_j[r] (deterministic)."""
        G = (C.c_double * (self.k * other.k))()
        with torch.cuda.device(self.dev):
            check(lib.femb_mv_gram(self.n, self.k, _p(self.data), self.n, other.k, _p(other.data), other.n, _p(w), G, _stream(self.dev)),
                  "femb_mv_gram")
        return torch.tensor(list(G), dtype=torch.float64).reshape(self.k, other.k)

    def update_into(self, coef, out, beta=0.0):
        """out_j = beta out_j + sum_i self_i coef[i][j]; `out` may be this object (in-place rotation / scaling)."""
        coef = torch.as_tensor(coef, dtype=torch.float64).reshape(self.k, out.k)
        Ch = _host_doubles(coef.reshape(-1).tolist())
        with torch.cuda.device(self.dev):
            check(lib.femb_mv_update(self.n, self.k, _p(self.data), self.n, out.k, Ch, float(beta), _p(out.data), out.n, _stream(self.dev)),
                  "femb_mv_update")
        return out

    def scale_mask(self, scale=None, mask=None):
        with torch.cuda.device(self.dev):
            check(lib.femb_mv_scale_mask(self.n, self.k, _p(self.data), self.n, _p(scale), _p(mask), _stream(self.dev)), "femb_mv_scale_mask")
        return self


# ----------------------------------------------------------------------------- 3x3 block-CSR (3-dof operators)

class Bsr3:
    """Operator with 3 dofs per node in block-CSR form: (brow int32 [nb+1], bcol int32 [nnzb], bval fp64 [nnzb,3,3])."""

    def __init__(self, brow, bcol, bval):
        self.brow, self.bcol, self.bval = brow, bcol, bval
        self.nb, self.nnzb, self.dev = brow.numel() - 1, bcol.numel(), bval.device

    @classmethod
    def from_csr_values(cls, brow, bcol, csr_val):
        """csr_val: values of the ndof=3 CSR generated from the node pattern (CsrPlan.pattern(3) / assemble(K, 3))."""
        assert csr_val.numel() == 9 * bcol.numel(), (csr_val.numel(), bcol.numel())
        bval = torch.empty((bcol.numel(), 3, 3), device=csr_val.device, dtype=torch.float64)
        with torch.cuda.device(csr_val.device):
            check(lib.femb_csr_bsr3_convert(1, brow.numel() - 1, _p(brow), _p(csr_val), _p(bval), _stream(csr_val.device)),
                  "femb_csr_bsr3_convert")
        return cls(brow, bcol, bval)

    def to_csr_values(self):
        out = torch.empty(9 * self.nnzb, device=self.dev, dtype=torch.float64)
        with torch.cuda.device(self.dev):
            check(lib.femb_csr_bsr3_convert(0, self.nb, _p(self.brow), _p(self.bval), _p(out), _stream(self.dev)), "femb_csr_bsr3_convert")
        return out

    def spmv(self, x):
        xx = x.to(device=self.dev, dtype=torch.float64).reshape(-1).contiguous()
        assert xx.numel() == 3 * self.nb
        y = torch.empty(3 * self.nb, device=self.dev, dtype=torch.float64)
        with torch.cuda.device(self.dev):
            check(lib.femb_spmv_bsr3(self.nb, self.nnzb, _p(self.brow), _p(self.bcol), _p(self.bval), _p(xx), _p(y), _stream(self.dev)),
                  "femb_spmv_bsr3")
        return y.reshape(x.shape)

    def jacobi(self, mask=None):
        out = torch.empty(3 * self.nb, device=self.dev, dtype=torch.float64)
        with torch.cuda.device(self.dev):
            check(lib.femb_bsr3_jacobi(self.nb, _p(self.brow), _p(self.bcol), _p(self.bval), _p(mask), _p(out), _stream(self.dev)),
                  "femb_bsr3_jacobi")
        return out

    def cg_solve(self, F, mask=None, minv=None, u_init=None, tol=1e-10, max_iter=1000, eps=1e-30, check_every=16):
        n = 3 * self.nb
        Ff = F.to(device=self.dev, dtype=torch.float64).reshape(-1).contiguous()
        assert Ff.numel() == n, (Ff.numel(), n)
        u = torch.zeros(n, device=self.dev, dtype=torch.float64) if u_init is None else \
            u_init.to(device=self.dev, dtype=torch.float64).reshape(-1).clone().contiguous()
        work = torch.empty(4 * n, device=self.dev, dtype=torch.float64)
        res = CGResult()
        with torch.cuda.device(self.dev):
            check(lib.femb_cg_solve_bsr3(self.nb, self.nnzb, _p(self.brow), _p(self.bcol), _p(self.bval), _p(Ff), _p(mask), _p(minv), _p(u),
                                         _p(work), float(tol), int(max_iter), float(eps), int(check_every), C.byref(res),
                                         _stream(self.dev)), "femb_cg_solve_bsr3")
        info = {"iterations": res.iterations, "status": STATUS.get(res.status, "?"), "rs": res.rs, "loop_ms": res.loop_ms}
        return u.reshape(F.shape), info
