"""ctypes binding of libfemb200.so (the C ABI declared in include/femb200.h).

The library is the ONLY compute path: there is no CPU fallback.  If the shared object is missing
the import fails loudly with the build command.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libfemb200.so")

c_i32, c_i64, c_f64, c_vp = C.c_int, C.c_int64, C.c_double, C.c_void_p


class CGResult(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("status", C.c_int32), ("rs", C.c_double), ("loop_ms", C.c_double),
                ("index_bytes", C.c_int32)]


# int (*femb_apply_fn)(void* ctx, const double* x, double* y, femb_stream stream)
APPLY_FN = C.CFUNCTYPE(C.c_int, c_vp, c_vp, c_vp, c_vp)

# name -> argtypes; every function returns int (status) unless listed in _RESTYPES
SIGNATURES = {
    "femb_version": [],
    "femb_elem_volumes": [c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp],
    "femb_c3d4": [c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, c_f64, c_f64, c_vp, c_vp, c_vp],
    "femb_solid": [c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, C.POINTER(c_f64), c_i32, c_f64, c_f64, c_vp, c_vp],
    "femb_default_points": [c_i32, C.POINTER(c_f64)],
    "femb_mass_points": [c_i32, C.POINTER(c_f64)],
    "femb_solid_stress": [c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, c_vp, C.POINTER(c_f64), c_i32, c_f64, c_f64, c_i32, c_vp, c_vp, c_vp],
    "femb_solid_geometric": [c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, c_vp, C.POINTER(c_f64), c_i32, c_f64, c_f64, c_vp, c_vp],
    "femb_shape_tables": [c_i32, C.POINTER(c_f64), c_i32, C.POINTER(c_f64), C.POINTER(c_f64)],
    "femb_stress_helper": [c_i32, c_vp, c_i32, c_i64, c_vp, c_vp],
    "femb_node_average": [c_vp, c_vp, c_i32, c_vp, c_vp],
    "femb_shell": [c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, C.POINTER(c_f64), c_i32, C.POINTER(c_f64), c_vp, c_vp],
    "femb_shell_ex": [c_i32, c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, C.POINTER(c_f64), c_i32, C.POINTER(c_f64), c_vp, c_vp, c_vp],
    "femb_shell_normal": [c_vp, c_i32, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp],
    "femb_shell_rotate_operator": [c_vp, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp],
    "femb_shell_local_coordinates": [c_vp, c_i32, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp],
    "femb_shell_local_displacement": [c_vp, c_i32, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp],
    "femb_shell_postprocess": [c_vp, c_i32, c_i64, c_i32, c_f64, c_f64, c_vp, c_vp],
    "femb_face_forces": [c_vp, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp],
    "femb_shared_face_forces_sum": [c_vp, c_i64, c_vp, c_i32, c_i32, c_vp, c_vp],
    "femb_wedge_face_normals": [c_vp, c_i32, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp],
    "femb_shell_extrude": [c_vp, c_vp, c_vp, c_i32, c_i64, c_f64, c_f64, c_vp, c_vp],
    "femb_extrude_connectivity": [c_vp, c_i32, c_i64, c_i32, c_i64, c_vp, c_vp],
    "femb_to_c3d4": [c_i32, c_vp, c_i32, c_i64, c_vp, c_vp],
    "femb_p2_create": [c_vp, c_i32, c_i64, c_i64, c_vp, C.POINTER(c_vp), C.POINTER(c_i64)],
    "femb_p2_fill": [c_vp, c_vp, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp],
    "femb_p2_destroy": [c_vp],
    "femb_entities_create": [c_i32, c_vp, c_i32, c_i64, c_i32, c_vp, C.POINTER(c_vp), C.POINTER(c_i64), C.POINTER(c_i64)],
    "femb_entities_surface": [c_vp, c_vp, c_vp, c_vp],
    "femb_entities_shared": [c_vp, c_vp, c_vp],
    "femb_entities_destroy": [c_vp],
    "femb_surface_normals": [c_vp, c_i32, c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp],
    "femb_face_normals_area": [c_i32, c_vp, c_i32, c_vp, c_i32, c_i64, c_i32, c_vp, c_vp],
    "femb_csr_plan_create": [c_vp, c_i32, c_i64, c_i32, c_i64, c_vp, C.POINTER(c_vp), C.POINTER(c_i64)],
    "femb_csr_plan_pattern": [c_vp, c_i32, c_vp, c_vp, c_vp],
    "femb_csr_assemble": [c_vp, c_i32, c_vp, c_vp, c_vp],
    "femb_csr_assemble_c3d4": [c_vp, c_i32, c_vp, c_f64, c_f64, c_vp, c_vp, c_vp],
    "femb_csr_plan_destroy": [c_vp],
    "femb_spmv": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_ebe_apply": [c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp],
    "femb_cg_solve": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f64, c_i32, c_f64, c_i32,
                      C.POINTER(CGResult), c_vp],
    "femb_cg_solve_bsr3": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_f64, c_i32, c_f64, c_i32,
                           C.POINTER(CGResult), c_vp],
    "femb_spmv_bsr3": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_csr_bsr3_convert": [c_i32, c_i64, c_vp, c_vp, c_vp, c_vp],
    "femb_bsr3_jacobi": [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_cg_solve_multi": [c_i64, c_i32, C.POINTER(c_i64), C.POINTER(c_vp), C.POINTER(c_vp), C.POINTER(c_vp), c_vp, c_vp, c_vp, c_vp,
                            c_vp, c_f64, c_i32, c_f64, c_i32, C.POINTER(CGResult), c_vp],
    "femb_cg_solve_operator": [c_i64, APPLY_FN, c_vp, c_vp, c_vp, c_vp, c_f64, c_i32, c_i32, C.POINTER(CGResult), c_vp],
    "femb_vtk_open": [C.c_char_p, C.POINTER(c_vp), C.POINTER(c_i64), C.POINTER(c_i64), C.POINTER(c_i64), C.POINTER(C.c_int32)],
    "femb_vtk_read": [c_vp, c_vp, c_vp, c_vp],
    "femb_vtk_close": [c_vp],
    "femb_ebe_diag": [c_vp, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp],
    "femb_mv_gram": [c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, C.POINTER(c_f64), c_vp],
    "femb_mv_update": [c_i64, c_i32, c_vp, c_i64, c_i32, C.POINTER(c_f64), c_f64, c_vp, c_i64, c_vp],
    "femb_mv_scale_mask": [c_i64, c_i32, c_vp, c_i64, c_vp, c_vp, c_vp],
    "femb_spmm_bsr3": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp],
    "femb_mb_gram": [c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp],
    "femb_mb_combine": [c_i64, c_i32, c_vp, c_i64, c_i32, C.POINTER(c_f64), c_f64, c_vp, c_i64, c_vp],
    "femb_lobpcg_residual": [c_i64, c_i32, c_vp, c_i64, c_vp, c_vp, c_i64, C.POINTER(c_f64), c_vp, c_i32, c_vp, c_vp, c_i64, c_vp, c_vp],
    "femb_mg_smooth_bsr3": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_f64, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp],
    "femb_mg_transfer": [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp],
    "femb_mg_transfer_bsr3": [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i64, c_i32, c_vp, c_i64, c_vp],
    "femb_amg_aggregate": [c_i64, c_vp, c_vp, c_vp, c_vp, C.POINTER(c_i64), c_vp],
    "femb_amg_tentative": [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_f64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_bsr3_spgemm": [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.POINTER(c_i64), c_vp],
    "femb_bsr3_transpose": [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_csr_jacobi": [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_graph_from_pairs": [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_vp],
    "femb_subdomain_forces": [c_vp, c_i32, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp],
    "femb_graph_bfs": [c_vp, c_vp, c_i64, c_vp, c_i32, c_vp, c_vp, C.POINTER(c_i32), c_vp],
    "femb_dist_header_bytes": [],
    "femb_dist_alloc": [c_i64, C.POINTER(c_vp), c_vp],
    "femb_dist_open": [c_vp, C.POINTER(c_vp)],
    "femb_dist_close": [c_vp],
    "femb_dist_free": [c_vp],
    "femb_dist_reset": [c_vp, c_vp],
    "femb_dist_cg_solve": [c_i32, c_i32, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.POINTER(c_vp), c_i32,
                           C.POINTER(C.c_int32), C.POINTER(C.c_int32), c_vp, C.POINTER(c_i64), c_vp, c_vp, c_vp, c_f64, c_i32, c_f64, c_i32,
                           c_i32, C.POINTER(CGResult), c_vp],
}
_RESTYPES = {"femb_last_error": C.c_char_p}


class FembError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C <package>/csrc`).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.femb_last_error.restype = C.c_char_p
    lib.femb_last_error.argtypes = []
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library out of sync
        fn.argtypes = args
        fn.restype = C.c_int
    return lib


lib = _load()


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib.femb_last_error().decode("utf-8", "replace")
        raise FembError(f"{what} failed (status {rc}): {msg}")
