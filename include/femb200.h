/*
 * libfemb200 -- C ABI of the B200-native (sm_100a) FEM hot path.
 *
 * The reference (sml2004/CUDA-powered-mesh-handling-and-Iterative-solvers) has no FFI: its boundary
 * is the module-level Python API of solver/element.py, solver/shell.py and solver/solver.py.  Each
 * entry point below names the reference function (file:line under /root/reference/solver/) whose torch
 * op chain it replaces; the Python mirror in <package>/solver/ binds them with ctypes (INTEGRATION.md).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host; tensors are contiguous row-major
 *  - `fp` = 4 (float) or 8 (double) bytes per real; `ib` = 4 (int32) or 8 (int64) bytes per index
 *  - the library never allocates user-visible memory: the caller passes outputs; data-dependent sizes use
 *    a plan handle (create -> query counts -> fill -> destroy); scratch comes from the stream-ordered pool
 *  - every call is asynchronous on `stream` (a cudaStream_t) unless it returns a count to the host
 *  - return value 0 = ok; otherwise femb_last_error() holds a message (thread-local)
 */
#ifndef FEMB200_H
#define FEMB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* femb_stream; /* cudaStream_t */

enum {
  FEMB_OK = 0,
  FEMB_ERR_ARG = 1,
  FEMB_ERR_CUDA = 2,
  FEMB_ERR_SINGULAR = 3, /* reference raises ValueError (element.py:857-858) */
  FEMB_ERR_NCCL = 4,
  FEMB_ERR_UNSUPPORTED = 5
};

const char* femb_last_error(void);
int femb_version(void);

/* ---------------------------------------------------------------------------------------------
 * Element kernels (solver/element.py)
 * ------------------------------------------------------------------------------------------- */

/* element kinds */
enum { FEMB_C3D4 = 4, FEMB_C3D6 = 6, FEMB_C3D8 = 8, FEMB_C3D10 = 10, FEMB_C3D15 = 15, FEMB_C3D20 = 20, FEMB_S3 = 103, FEMB_S4 = 104 };

/* compute_tetrahedral_volumes :514-541, compute_hexahedral_volumes :1248-1291, compute_wedge_volumes :2198-2232.
 * vol[M] = sum of |det|/6 over the reference's sub-tet table of `kind`. */
int femb_elem_volumes(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, int conn_stride,
                      void* vol, femb_stream stream);

/* compute_c3d4_B_matrix :835-881 (what = 0: gradients [M,4,3]; 1: B [M,6,12]) and compute_c3d4_K_matrix :883-903
 * (what = 2: K [M,12,12] = B^T D B V; 3: Poisson V G G^T [M,4,4] (not in the reference); 4: consistent mass
 * rho V/20 (1+delta) (x) I3 [M,12,12] with rho passed in `E` (not in the reference)).
 * `flag` (device int32, zeroed by the caller) is set to 1 when any |det[1,x,y,z]| < 1e-12 (-> ValueError). */
int femb_c3d4(int what, const void* coords, int fp, const void* conn, int ib, int64_t M, double E, double nu, void* out,
              int32_t* flag, femb_stream stream);

/* Isoparametric solids C3D10/C3D8/C3D6/C3D20/C3D15:
 *   compute_c3d10_{Jacobian,shape_gradients,B_matrix,K_matrix} :1026-1125,:1191-1239
 *   compute_c3d8_*  :1601-1694,:1754-1803     compute_c3d6_* :2482-2568,:2631-2676
 *   compute_c3d20_* :1921-2188 (the reference's Jacobian raises and its derivative table is wrong; this is the
 *   standard 20-node serendipity hex in VTK/Abaqus node order) and C3D15 (dispatch targets :377-426 are undefined
 *   in the reference; standard 15-node wedge) -- both "parity unpinned", validated by invariants.
 * `pts_host` = [nq,4] doubles (xi,eta,zeta,w) on the HOST (the caller resolves defaults; the library ships
 * the reference's rules through femb_default_points).
 * what = 0: J [M,3,3] at pts[0]; 1: gradients [M,nen,3] at pts[0]; 2: B [M,6,3nen] at pts[0];
 *        3: K [M,nd,nd] = sum_q w_q detJ_q B^T D B (signed detJ);
 *        4: per-point K [nq,M,nd,nd] = detJ_q B^T D B, unweighted (single=False);
 *        5: (C3D6 single=True) K = B^T D B at pts[0] times the 3-tet |volume|;
 *        6: consistent mass [M,nd,nd] = rho sum_q w_q |detJ_q| N^T N (x) I3 with rho passed in `E` (the reference only
 *           calls an undefined compute_c3d4_M_matrix, solver_example.ipynb cell 13 -- parity unpinned). */
int femb_solid(int kind, int what, const void* coords, int fp, const void* conn, int ib, int64_t M, const double* pts_host,
               int nq, double E, double nu, void* out, femb_stream stream);

/* c3d10_integration_points :995-1024, c3d8_integration_points :1583-1599, c3d6_integration_points :2448-2480,
 * c3d20_integration_points :1898-1919, s4_integration_points shell.py:651-672; C3D15: 3-point triangle x 3-point Gauss
 * (not in the reference).  Fills pts_host[nq*4] (shells: xi,eta,0,w), returns nq (or -1). */
int femb_default_points(int kind, double* pts_host);

/* Rules used by the consistent mass (what = 6) when the caller passes none: C3D10 degree-5 14-point, C3D8/C3D20
 * 3x3x3 Gauss, C3D6/C3D15 degree-4 triangle x 3-point Gauss.  Fills pts_host[nq*4], returns nq <= 27 (or -1). */
int femb_mass_points(int kind, double* pts_host);

/* Host-only: the natural-coordinate tables the solid kernels consume, N_host[nq,nen] and dN_host[nq,nen,3] at the
 * points pts_host[nq,4] (the host part of compute_*_Jacobian's dN_dnatural, e.g. element.py:1042-1055). */
int femb_shape_tables(int kind, const double* pts_host, int nq, double* N_host, double* dN_host);

/* Stress recovery: compute_c3d4_element_stress :905-939, compute_c3d10_element_stress :1127-1189,
 * compute_c3d8_element_stress :1696-1752, compute_c3d6_element_stress :2570-2629 (+ C3D20 / C3D15).
 * disp[N,3]; single != 0: stress[M,3,3] = sum_q w_q sigma_q and vm[M] = sum_q w_q vonMises(sigma_q);
 * single == 0: stress[nq,M,3,3], vm[nq,M].  C3D4 takes one point with weight 1. */
int femb_solid_stress(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, const void* disp,
                      const double* pts_host, int nq, double E, double nu, int single, void* stress, void* vm,
                      femb_stream stream);

/* Geometric stiffness of the stress state of a displacement field (not in the reference).
 * kind = FEMB_C3D4 (one point, pts ignored) or FEMB_C3D10 (pts_host [nq,4] on the host, 1 <= nq <= 16; other kinds -> error).
 * disp [N,3] in the precision of coords.  At every point q: eps = sym(sum_c u_c (x) g_c), sigma = lam tr(eps) I + 2 mu eps,
 * s_ab = sum_q w_q |detJ_q| g_a^T sigma_q g_b;  out [M, 3nen, 3nen] with block (a,b) = s_ab I3 (bitwise symmetric). */
int femb_solid_geometric(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, const void* disp,
                         const double* pts_host, int nq, double E, double nu, void* out, femb_stream stream);

/* Shell elements (solver/shell.py): compute_s3_* :297-453, compute_s4_* :597-861.
 * what = 0: unit [M,3,3]; 1: J [M,2,2]; 2: gradients [M,nen,2]; 3: B [M,6,6nen]; 4: K [M,6nen,6nen];
 *        5: (S4) per-point K [M,24,24,nq] (single=False).  S3 ignores pts. D6 = Kirchhoff D as 36 doubles (host). */
int femb_shell(int kind, int what, const void* coords, int fp, const void* conn, int ib, int64_t M, const double* pts_host,
               int nq, const double* D6_host, void* out, femb_stream stream);

/* Extended shell entry.  fac_host[nq,5] = (1-xi, 1+xi, 1-eta, 1+eta, w): the four bilinear factors are passed evaluated
 * because the reference forms them in the dtype of what it was handed -- python doubles on the K path (shell.py:841-842),
 * 0-dim fp32 tensors when compute_s4_B_matrix iterates over its fp32 rule (:813-814 -> :683-695).  S3 ignores fac_host.
 * what 0..5 as femb_shell, plus
 *   7: sum_q w_q B_q [M,6,6nen]   8: per-point w_q B_q [M,6,6nen,nq]   (compute_s4_B_matrix :802-823)
 *   9: stress resultants [M,6] = D (sum_q w_q B_q) disp[conn] with disp [N,6] in GLOBAL axes exactly as the reference takes it
 *      (compute_s3_shell_stress :455-481, compute_s4_shell_stress :863-879) */
int femb_shell_ex(int kind, int what, const void* coords, int fp, const void* conn, int ib, int64_t M, const double* fac_host,
                  int nq, const double* D6_host, const void* disp, void* out, femb_stream stream);

/* compute_s3_global_to_local_coordinates shell.py:323-347, compute_s4_global_to_local_coordinates :625-649:
 * out[M,nen,3] = coordinates relative to node 0 of each element expressed in the frame unit[M,3,3] (rows = axes) */
int femb_shell_local_coordinates(const void* coords, int fp, const void* conn, int ib, int64_t M, int nen, const void* unit, void* out,
                                 femb_stream stream);

/* compute_s3_normal shell.py:184-203 (nen = 3: cross(x1-x0, x2-x0)/2) and compute_s4_normal :483-502 (nen = 4:
 * cross(x1-x0, x3-x0)): out[M,3] */
int femb_shell_normal(const void* coords, int fp, const void* conn, int ib, int64_t M, int nen, void* out, femb_stream stream);
/* Shell element operator in global axes: out[M,nd,nd] = T^T K T, T = blockdiag(unit, unit, ...) per 3 dofs -- the operator
 * compute_shell_nodal_forces (shell.py:58-102) applies by rotating in and out of the element frame; assembled once for the
 * shell CG (solver.py:297-389) and the shell families of static_structure_solver (:11-135). */
int femb_shell_rotate_operator(const void* K, const void* unit, int fp, int64_t M, int nd, void* out, femb_stream stream);

/* compute_global_to_local_displacement shell.py:41-56: out[M,nen,6] = (unit g_trans, unit g_rot), g = disp[conn] ([N,6]) */
int femb_shell_local_displacement(const void* conn, int ib, int64_t M, int nen, const void* disp, const void* unit, int fp,
                                  void* out, femb_stream stream);

/* compute_shell_postprocess_values shell.py:104-160: nmq[M,ncol] (N, M resultants in columns 0..5) -> out[8,M] =
 * sx, sy, txy, s1, s2, theta_p, tau_max, vm at through-thickness coordinate z of a shell of thickness t */
int femb_shell_postprocess(const void* nmq, int fp, int64_t M, int ncol, double t, double z, void* out, femb_stream stream);

/* compute_c3d4_surface_forces element.py:3343-3360: out[M,nf,3] = stress[M,3,3] normals[M,nf,3] */
int femb_face_forces(const void* normals, const void* stress, int fp, int64_t M, int nf, void* out, femb_stream stream);
/* compute_c3d4_shared_face_forces_sum element.py:3362-3384: out[S,3] = forces[e1,f1] + forces[e2,f2], pairs[S,2,2] int64 */
int femb_shared_face_forces_sum(const int64_t* pairs, int64_t S, const void* forces, int fp, int nf, void* out, femb_stream stream);

/* compute_stress_tensor :308-330 (what = 0: Voigt [M,6] xx,yy,zz,xy,yz,zx -> [M,3,3]) and compute_von_mises_stress
 * :332-353 (what = 1: [M,3,3] -> [M]). */
int femb_stress_helper(int what, const void* in, int fp, int64_t M, void* out, femb_stream stream);

/* Fixed-table connectivity expansion: c3d10_to_c3d4 :963-993, c3d8_to_c3d4 :1555-1581, c3d6_to_c3d4 :2424-2446,
 * c3d20_to_c3d4 :1852-1896.  out[k*M,4] int64, k = 8/6/3/24. */
int femb_to_c3d4(int kind, const void* conn, int ib, int64_t M, int64_t* out, femb_stream stream);

/* c3d4_to_c3d10 :777-833 (P1 -> P2 mid-edge insertion; the reference is a Python dict loop).  New node ids are handed out
 * in first-encounter order over (element-major, edge slots (0,1),(1,2),(2,0),(0,3),(1,3),(2,3)): bit-exact numbering.
 * Count-then-fill: create returns the number of distinct edges E; fill writes conn10[M,10] int32, coords_out[N+E,3]
 * (fp_out = 4 or 8; mid points are (x_lo + x_hi) / 2) and edges[E,2] int32 = the end points behind new node N + r (used
 * by the caller to grow its RBE2 / RBE3 node sets).  Any of the three outputs may be NULL. */
typedef struct femb_p2_plan femb_p2_plan;
int femb_p2_create(const void* conn, int ib, int64_t M, int64_t n_nodes, femb_stream stream, femb_p2_plan** plan, int64_t* n_edges);
int femb_p2_fill(femb_p2_plan* plan, const void* conn, int ib, const void* coords, int fp_in, int fp_out, int32_t* conn10,
                 void* coords_out, int32_t* edges, femb_stream stream);
int femb_p2_destroy(femb_p2_plan* plan);

/* ---------------------------------------------------------------------------------------------
 * Topology (bit-exact): faces of solids, edges of shells
 *   surface: compute_tetrahedral_surface_faces_with_fourth_node :543-579, hex :1293-1334, wedge :2234-2283,
 *            shell.py compute_triangle_surface_faces_with_third_node :261-295, square :561-597
 *   shared : identify_tetrahedral_shared_faces :707-762, hex :1474-1532, shell.py S3 :205-259, S4 :504-559
 * ------------------------------------------------------------------------------------------- */
enum {
  FEMB_ENT_TET_FACES = 0,
  FEMB_ENT_HEX_FACES = 1,
  FEMB_ENT_WEDGE_QUADS = 2,
  FEMB_ENT_WEDGE_TRIS = 3,
  FEMB_ENT_TRI_EDGES = 4,
  FEMB_ENT_QUAD_EDGES = 5
};
typedef struct femb_entity_plan femb_entity_plan;
/* Sorts the canonical (ascending) node tuples of all entities once; synchronises the stream to return counts. */
int femb_entities_create(int ent_kind, const void* conn, int ib, int64_t M, int conn_stride, femb_stream stream,
                         femb_entity_plan** plan, int64_t* n_surface, int64_t* n_shared);
/* faces[K,nfn] int64 in slot-major order with the element's node order, extra[K] = off-entity node */
int femb_entities_surface(femb_entity_plan* plan, int64_t* faces, int64_t* extra, femb_stream stream);
/* pairs[S,2,2] int64 = ((elem,local),(elem,local)), rows lexicographic by sorted tuple, lower element id first.
 * `pairs` must be 32-byte aligned (each row leaves as one 32-byte store). */
int femb_entities_shared(femb_entity_plan* plan, int64_t* pairs, femb_stream stream);
int femb_entities_destroy(femb_entity_plan* plan);

/* Outward normals: compute_tetrahdral_surface_normals :581-619, hex :1336-1374, wedge :2285-2338.
 * faces[K,nfn] + extra[K] as returned above; `second` = which face node forms the second edge (2; wedge quads 3). */
int femb_surface_normals(const void* coords, int fp, const int64_t* faces, const int64_t* extra, int64_t K, int nfn,
                         int second, void* normals, femb_stream stream);
/* compute_tetrahedral_normals_and_area :652-705 (kind=FEMB_C3D4, [M,4,3]),
 * compute_hexahedral_normals_and_area :1418-1472 (kind=FEMB_C3D8, [M,6,3]) */
int femb_face_normals_area(int kind, const void* coords, int fp, const void* conn, int ib, int64_t M, int conn_stride,
                           void* out, femb_stream stream);

/* compute_wedge_normals_and_area :2377-2420: UNIT normals [M,5,3] of the faces (0,1,4,3) (1,2,5,4) (2,0,3,5) (0,2,1) (3,4,5),
 * not re-oriented (the reference neither orients nor area-weights them, despite the name) */
int femb_wedge_face_normals(const void* coords, int fp, const void* conn, int ib, int64_t M, int conn_stride, void* out,
                            femb_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Global assembly: COO (subdivision.ipynb cell 6) -> CSR, deterministic
 * ------------------------------------------------------------------------------------------- */
typedef struct femb_csr_plan femb_csr_plan;
/* Builds the node-level sparsity pattern and the node->element incidence lists (sort based).
 * n_nodes = elements.max()+1 as in cell 6 line 11.  Synchronises the stream to return nnz_nodes. */
int femb_csr_plan_create(const void* conn, int ib, int64_t M, int nen, int64_t n_nodes, femb_stream stream,
                         femb_csr_plan** plan, int64_t* nnz_nodes);
/* dof-level pattern for `ndof` dofs per node: crow[n_nodes*ndof+1], col[nnz_nodes*ndof^2] (int32), identical to
 * torch.sparse_coo_tensor(...).coalesce().to_sparse_csr() of the cell-6 COO. */
int femb_csr_plan_pattern(femb_csr_plan* plan, int ndof, int32_t* crow, int32_t* col, femb_stream stream);
/* vals[nnz] (fp64) = ordered (element-ascending) sums of the materialised element matrices Ke[M,nen*ndof,nen*ndof] */
int femb_csr_assemble(femb_csr_plan* plan, int ndof, const double* Ke, double* vals, femb_stream stream);
/* fused P1-tet assembly straight from coordinates (never materialises Ke): kind 0 = Poisson (ndof 1),
 * 1 = elasticity (ndof 3, E/nu). */
int femb_csr_assemble_c3d4(femb_csr_plan* plan, int kind, const double* coords, double E, double nu, double* vals,
                           int32_t* flag, femb_stream stream);
int femb_csr_plan_destroy(femb_csr_plan* plan);

/* ---------------------------------------------------------------------------------------------
 * Operator application and Krylov solvers
 * ------------------------------------------------------------------------------------------- */
/* y = A x, CSR with int32 indices and fp64 values */
int femb_spmv(int64_t n_rows, int64_t nnz, const int32_t* crow, const int32_t* col, const double* val, const double* x, double* y,
              femb_stream stream);

/* compute_nodal_forces element.py:429-464: y[N,ndof] = sum_e K_e u_e, deterministic (incidence ordered).
 * compute_shell_nodal_forces shell.py:58-102 when unit != NULL (ndof = 6, rotates into/out of the element frame). */
int femb_ebe_apply(femb_csr_plan* plan, int ndof, const void* Ke, const void* u, const void* unit, int fp, void* y,
                   femb_stream stream);

/* shell_extrude shell.py:885-983: per-node unit normals of a mid-surface mesh (mean of the unit normals of the incident
 * triangles and of both triangles (0,1,2), (0,2,3) of the incident quads, eps = 1e-8 in every denominator), then
 * coords3d[2N,3] = (x - t/2 n | x + t/2 n).  tri / quad = plans of the [T,3] / [S,4] connectivity built with n_nodes = N
 * (either may be NULL); sums run over the incidence lists in the reference's order (deterministic). */
int femb_shell_extrude(femb_csr_plan* tri, femb_csr_plan* quad, const void* coords, int fp, int64_t N, double thickness, double eps,
                       void* coords3d, femb_stream stream);
/* out[M,2nen] = (conn | conn + N): wedges from triangles, hexahedra from quads (shell.py:957-973); same index type */
int femb_extrude_connectivity(const void* conn, int ib, int64_t M, int nen, int64_t N, void* out, femb_stream stream);

/* Diagonal of sum_e K_e without assembling: out[N*ndof], element-ascending sums.  Lumped mass of vectorized_modal_solver
 * (solver.py:1126-1131) and the Jacobi diagonal behind compute_diagonal_preconditioner (solver.py:814-833); col0 != 0 sums
 * column 0 of every element row instead (the reference preconditioner's strided-view bug, solver.py:828). */
int femb_ebe_diag(femb_csr_plan* plan, int ndof, const void* Ke, int fp, int col0, void* out, femb_stream stream);

/* compute_node_vm_stress element.py:466-504: out[N] = mean over the elements containing the node of elem_values[M]
 * (0 for nodes without elements); sums run in ascending element order (deterministic; the reference uses index_add). */
int femb_node_average(femb_csr_plan* plan, const void* elem_values, int fp, void* out, femb_stream stream);

/* Block-CSR with 3x3 blocks for 3-dof operators (every elasticity operator of the reference: dofs = node*3+{0,1,2},
 * element.py:447-449).  brow[nb+1] / bcol[nnzb] = the node-level pattern (femb_csr_plan_pattern with ndof = 1),
 * bval[nnzb][3][3] row-major.  8.44 instead of 12 bytes per scalar nonzero and a third of the x gathers.
 *   femb_csr_bsr3_convert: permutes between the ndof=3 CSR values of femb_csr_assemble and the block layout (to_bsr != 0
 *   CSR -> blocks, else blocks -> CSR); in and out must not alias.
 *   femb_spmv_bsr3: y = A x, x/y [3 nb].   femb_bsr3_jacobi: minv[3 nb] = 1/diag (0 for masked or zero-diagonal rows). */
int femb_csr_bsr3_convert(int to_bsr, int64_t nb, const int32_t* brow, const double* in, double* out, femb_stream stream);
int femb_spmv_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* bval, const double* x, double* y,
                   femb_stream stream);
int femb_bsr3_jacobi(int64_t nb, const int32_t* brow, const int32_t* bcol, const double* bval, const uint8_t* mask, double* minv,
                     femb_stream stream);

typedef struct femb_cg_result {
  int32_t iterations; /* the count the reference prints: i+1 at exit, max_iter when not converged */
  int32_t status;     /* 0 converged, 1 breakdown (pAp guard / NaN), 2 max_iter */
  double rs;          /* last r.r (or r.z) */
  double loop_ms;     /* device time of the iteration loop (CUDA events on the solver stream) */
  int32_t index_bytes; /* bytes per column index the loop's SpMV streamed: 2 = 16-bit delta-encoded, 4 = int32 CSR */
} femb_cg_result;

/* stable_conjugate_gradient_solver solver.py:144-229 (also the loops of :11-135, :231-295, :297-389) on the
 * assembled operator: projected CG, rows with mask[i]==0 are held at zero, absolute test sqrt(r.r)<tol,
 * +eps denominators, pAp guards.  minv != NULL selects preconditioned_conjugate_gradient_solver :766-812
 * (z = minv*r, test sqrt(r.z)<tol, no guards, no eps).  u holds u_init on entry and the solution on exit.
 * work = 4*n doubles of caller scratch.  The loop is captured in a CUDA graph; blocks until done. */
int femb_cg_solve(int64_t n, int64_t nnz, const int32_t* crow, const int32_t* col, const double* val, const double* F,
                  const uint8_t* mask, const double* minv, double* u, double* work, double tol, int max_iter, double eps,
                  int check_every, femb_cg_result* result_host, femb_stream stream);

/* Same loop on a 3x3 block-CSR operator (n = 3 nb unknowns; F, mask, minv, u, work sized as for femb_cg_solve). */
int femb_cg_solve_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* bval, const double* F,
                       const uint8_t* mask, const double* minv, double* u, double* work, double tol, int max_iter, double eps,
                       int check_every, femb_cg_result* result_host, femb_stream stream);

/* Same loop with the operator given as a SUM of up to 8 CSR matrices over the same n rows (static_structure_solver
 * solver.py:11-135 sums one operator per element family: C3D4/C3D8/C3D6 on the translations, S3/S4 on all six dofs).
 * The *_host arguments are host arrays of nmat device pointers / sizes. */
int femb_cg_solve_multi(int64_t n, int nmat, const int64_t* nnz_host, const int32_t* const* crow_host,
                        const int32_t* const* col_host, const double* const* val_host, const double* F, const uint8_t* mask,
                        const double* minv, double* u, double* work, double tol, int max_iter, double eps, int check_every,
                        femb_cg_result* result_host, femb_stream stream);

/* conjugate_gradient_solver_Ku solver.py:1029-1065: CG on an operator supplied as a function (no node fixing, no guards, no
 * eps; u must hold the start vector -- zeros in the reference -- and returns the solution).  `apply(ctx, x, y, stream)` must
 * enqueue y = K x on `stream` and return 0.  work = 3*n doubles.  The host reads the stop flag every check_every iterations. */
typedef int (*femb_apply_fn)(void* ctx, const double* x, double* y, femb_stream stream);
int femb_cg_solve_operator(int64_t n, femb_apply_fn apply, void* ctx, const double* R, double* u, double* work, double tol,
                           int max_iter, int check_every, femb_cg_result* result_host, femb_stream stream);

/* Tall-skinny kernels of the subspace-iteration modal solver (vectorized_modal_solver solver.py:1084-1312).  Vectors are stored
 * one after the other: column i of X at X + i*ldx (ldx >= n), 1 <= ki, kj <= 8.
 *   femb_mv_gram:   G_host[i*kj+j] = sum_r X_i[r] w[r] Y_j[r] (w = NULL: 1); deterministic two-stage sums; synchronises.
 *   femb_mv_update: Y_j = beta Y_j + sum_i X_i C_host[i*kj+j]; Y may alias X (in-place scaling / basis rotation).
 *   femb_mv_scale_mask: X_j[r] *= scale[r] (NULL: 1), set to 0 where mask[r] == 0 (NULL: nowhere). */
int femb_mv_gram(int64_t n, int ki, const double* X, int64_t ldx, int kj, const double* Y, int64_t ldy, const double* w, double* G_host,
                 femb_stream stream);
int femb_mv_update(int64_t n, int ki, const double* X, int64_t ldx, int kj, const double* C_host, double beta, double* Y, int64_t ldy,
                   femb_stream stream);
int femb_mv_scale_mask(int64_t n, int k, double* X, int64_t ldx, const double* scale, const uint8_t* mask, femb_stream stream);

/* Block kernels of the LOBPCG modal solver (lowest_modes, not in the reference).  Multivectors are ROW-MAJOR and node-interleaved:
 * value (dof r, column j) at X[r*ld + j], ld >= the columns used.  Sums are deterministic (fixed-order two-stage reductions, no
 * atomics); outputs must not overlap inputs (views of one buffer with the same ld and disjoint columns are allowed).
 *   femb_spmm_bsr3: YK = K X and, when mval != NULL, YM = M X in the same pass; K and M share brow/bcol (3x3 blocks as in
 *     femb_spmv_bsr3), 1 <= m <= 16 columns; mask (NULL: none) zeroes x and y on dofs with mask == 0.
 *   femb_mb_gram: G[i*kb+j] = sum_r A[r*lda+i] B[r*ldb+j], 1 <= ka, kb <= 48; G is a device array.
 *   femb_mb_combine: Y[:, :mc] = beta Y[:, :mc] + X[:, :k] C_host (C_host [k, mc] row-major), 1 <= k <= 48, 1 <= mc <= 16.
 *   femb_lobpcg_residual: r_j = KX_j - lam_host[j] MX_j for j < m (KX, MX share ldk); norms[j] = |r_j|^2, norms[m+j] = |X_j|^2;
 *     W[:, a] = dinv * r_{active[a]} for a < na (active: device int32 list). */
int femb_spmm_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* kval, const double* mval,
                   const uint8_t* mask, int m, const double* X, int64_t ldx, double* YK, double* YM, int64_t ldy, femb_stream stream);
int femb_mb_gram(int64_t n, int ka, const double* A, int64_t lda, int kb, const double* B, int64_t ldb, double* G, femb_stream stream);
int femb_mb_combine(int64_t n, int k, const double* X, int64_t ldx, int mc, const double* C_host, double beta, double* Y, int64_t ldy,
                    femb_stream stream);
int femb_lobpcg_residual(int64_t n, int m, const double* X, int64_t ldx, const double* KX, const double* MX, int64_t ldk,
                         const double* lam_host, const double* dinv, int na, const int32_t* active, double* W, int64_t ldw,
                         double* norms, femb_stream stream);

/* Multigrid V-cycle kernels of subdivided_lowest_modes (same multivector layout and rules as the block kernels above).
 *   femb_mg_smooth_bsr3: t = mask (R - A X_in) on 1 <= m <= 16 columns (A: 3x3 block-CSR as in femb_spmm_bsr3, x masked as there;
 *     mask NULL: none); Res = t and X_out = X_in + omega dinv t, each optional (at least one given; dinv [3 nb] needed with X_out).
 *     X_in NULL means X_in = 0 (X_out = omega dinv mask R, the matrix is not read).  X_out must not overlap X_in: ping-pong.
 *   femb_mg_transfer: Y[3i+d, j] (+)= mask_out[3i+d] sum_k val[k] X[3 col[k]+d, j] for the node-level scalar CSR (crow [n_out+1],
 *     col [nnz] < n_in, int32; val fp64) -- the prolongation or the restriction; accumulate = 1 adds to Y, 0 overwrites it. */
int femb_mg_smooth_bsr3(int64_t nb, int64_t nnzb, const int32_t* brow, const int32_t* bcol, const double* aval, const uint8_t* mask,
                        const double* dinv, double omega, int m, const double* R, int64_t ldr, const double* X_in, int64_t ldx,
                        double* X_out, int64_t ldo, double* Res, int64_t ldres, femb_stream stream);
int femb_mg_transfer(int64_t n_out, int64_t n_in, int64_t nnz, const int32_t* crow, const int32_t* col, const double* val,
                     const uint8_t* mask_out, int m, const double* X, int64_t ldx, int accumulate, double* Y, int64_t ldy,
                     femb_stream stream);

/* Smoothed-aggregation multigrid (femb200/amg.py): every level is a square 3x3 block-CSR operator, the transfers are rectangular
 * 3x3 block-CSR matrices (brow [rows+1], bcol int32, bval fp64 [nnzb, 3, 3]).  Aggregate a of the fine nodes gives the coarse
 * pseudo-nodes 2a (translation columns) and 2a+1 (rotation columns).  Results do not depend on thread scheduling.
 *   femb_mg_transfer_bsr3: Y[3i+d, j] (+)= mask_out[3i+d] (T X)[3i+d, j] for T with n_out block rows and block columns < n_in;
 *     layout and rules as femb_mg_transfer.
 *   femb_amg_aggregate: agg[nb] (int32) and *n_agg_host from the node graph (brow, bcol: a square block pattern); a node whose
 *     three dofs are masked (mask NULL: none) gets -1.  Distance-2 maximal independent set by synchronous rounds (priority: a
 *     fixed hash of the node id), roots take their neighbours, the rest join the neighbouring aggregate with the lowest id.
 *   femb_amg_tentative: the tentative prolongator of `agg` (n_agg aggregates): prow [nb+1] (two blocks per aggregated node),
 *     pcol / pval [2 n_aggregated], the coarse near-nullspace Bc [6 n_agg, 6] (global rigid-body modes), the coarse mask
 *     mask_c [6 n_agg] and the coarse node coordinates coords_c [2 n_agg, 3] (both pseudo-nodes at the aggregate's centroid).
 *     coords [nb, 3] are always given; the near-nullspace is the rigid-body modes of coords on the finest level (B NULL) and
 *     B [3 nb, 6] on coarser ones; masked rows are zero.  Per aggregate the rotation columns are re-centred on its centroid and
 *     scaled by 1 / its diameter, then CholQR2; a Cholesky pivot <= drop * (largest Gram diagonal) drops its column and masks its
 *     coarse dof.
 *   femb_bsr3_spgemm: C = X Y, X with n_rows block rows.  Call it twice: with ccol = cval = NULL it writes crow [n_rows+1] and
 *     *nnz_host; then with ccol [nnz], cval [nnz, 3, 3] (and xval, yval) it writes the sorted columns and the values.  A row of
 *     C may hold at most 2048 blocks: a wider row returns FEMB_ERR_UNSUPPORTED.
 *   femb_bsr3_transpose: R = P^T (rrow [n_cols+1], rcol / rval [nnzb]), blocks transposed, each row of R in increasing column. */
int femb_mg_transfer_bsr3(int64_t n_out, int64_t n_in, int64_t nnzb, const int32_t* trow, const int32_t* tcol, const double* tval,
                          const uint8_t* mask_out, int m, const double* X, int64_t ldx, int accumulate, double* Y, int64_t ldy,
                          femb_stream stream);
int femb_amg_aggregate(int64_t nb, const int32_t* brow, const int32_t* bcol, const uint8_t* mask, int32_t* agg, int64_t* n_agg_host,
                       femb_stream stream);
int femb_amg_tentative(int64_t nb, int64_t n_agg, const int32_t* agg, const uint8_t* mask, const double* coords, const double* B,
                       double drop, int32_t* prow, int32_t* pcol, double* pval, double* Bc, uint8_t* mask_c, double* coords_c,
                       femb_stream stream);
int femb_bsr3_spgemm(int64_t n_rows, const int32_t* xrow, const int32_t* xcol, const double* xval, const int32_t* yrow,
                     const int32_t* ycol, const double* yval, int32_t* crow, int32_t* ccol, double* cval, int64_t* nnz_host,
                     femb_stream stream);
int femb_bsr3_transpose(int64_t n_rows, int64_t n_cols, int64_t nnzb, const int32_t* prow, const int32_t* pcol, const double* pval,
                        int32_t* rrow, int32_t* rcol, double* rval, femb_stream stream);

/* Jacobi diagonal of a CSR matrix: minv[i] = mask[i] ? 1/A_ii : 0 (the documented replacement for the
 * reference's broken compute_diagonal_preconditioner solver.py:814-833) */
int femb_csr_jacobi(int64_t n, const int32_t* crow, const int32_t* col, const double* val, const uint8_t* mask,
                    double* minv, femb_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Element-graph partition (subdivision.ipynb cells 8-9: build_adjacency_matrix, pick_distant_seeds,
 * region_growing_partition)
 * ------------------------------------------------------------------------------------------- */
/* Symmetric CSR adjacency of M vertices from S undirected pairs.  pairs: int64, vertex ids at [t*pair_stride] and
 * [t*pair_stride + pair_stride/2] -- pair_stride = 4 reads the [S,2,2] output of femb_entities_shared directly (element
 * ids at 0 and 2), pair_stride = 2 a plain [S,2] list.  crow[M+1], col[2S], neighbours ascending.  Synchronises. */
int femb_graph_from_pairs(const int64_t* pairs, int64_t S, int pair_stride, int64_t M, int32_t* crow, int32_t* col,
                          femb_stream stream);
/* Level-synchronous multi-source BFS: dist[M] (hops to the nearest source, -1 unreachable) and, when label != NULL,
 * label[M] = index (into sources) of the region that reached the vertex first, highest index on ties.  One kernel per
 * level; the host reads one flag per level.  levels_host (optional) receives the number of levels.  Synchronises. */
int femb_graph_bfs(const int32_t* crow, const int32_t* col, int64_t M, const int64_t* sources, int n_sources, int32_t* dist,
                   int32_t* label, int32_t* levels_host, femb_stream stream);

/* subdivision.ipynb cell 15 (make_sub_domain_forces): out[n_sub,N,3] = F[N,3] copied to every subdomain, then for each of the
 * ntgt interface targets o = tgt[t] = sub*N + node (unique): out[o] = F[node] + (fv[plus[t]] - fv[minus[t]]), an index of -1
 * meaning "absent" (first / last subdomain of the node's group).  free_vars [n_free,3] in the dtype of F. */
int femb_subdomain_forces(const void* F, int fp, int64_t N, int n_sub, const void* free_vars, int64_t ntgt, const int64_t* tgt,
                          const int32_t* plus, const int32_t* minus, void* out, femb_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Mesh input: legacy .vtk unstructured grids (vtk_loader_to_torch element.py:39-90 reads them through pyvista)
 * ------------------------------------------------------------------------------------------- */
typedef struct femb_vtk_mesh femb_vtk_mesh;
/* Parses the file on the host (ASCII or BINARY; classic CELLS and the 5.x OFFSETS/CONNECTIVITY layout).  cells_size = length
 * of the flat `[nen, id0, .., nen, id0, ..]` array (= pyvista's mesh.cells); points_are_float = file stores 32-bit reals. */
int femb_vtk_open(const char* path, femb_vtk_mesh** mesh, int64_t* n_points, int64_t* n_cells, int64_t* cells_size,
                  int32_t* points_are_float);
/* Copies into caller-owned HOST arrays: points_host[n_points*3], cells_host[cells_size], types_host[n_cells] (any may be NULL) */
int femb_vtk_read(femb_vtk_mesh* mesh, double* points_host, int64_t* cells_host, int32_t* types_host);
int femb_vtk_close(femb_vtk_mesh* mesh);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU CG over NVLink peer memory (one process per GPU; nothing to match in the reference, SURVEY 8e)
 * ------------------------------------------------------------------------------------------- */
/* Each rank allocates one "symmetric" buffer = header (femb_dist_header_bytes) + p[n_owned+n_ghost] doubles with
 * femb_dist_alloc, publishes the 64-byte cudaIpc handle to its peers (any side channel, e.g. torch.distributed),
 * and maps every peer's buffer with femb_dist_open. */
int femb_dist_header_bytes(void);
int femb_dist_alloc(int64_t bytes, void** ptr, void* ipc_handle64);
int femb_dist_open(const void* ipc_handle64, void** ptr);
int femb_dist_close(void* ptr);
int femb_dist_free(void* ptr);
int femb_dist_reset(void* own_sym, femb_stream stream); /* zero the flags; callers barrier across ranks afterwards */

/* The reference's projected CG (solver.py:144-229) / Jacobi-PCG (:766-812, minv != NULL) on row-partitioned data.
 * Local operator = owned rows only, columns in local numbering [owned | ghost]; F, mask, minv, u are owned-only.
 *   block = 1: scalar CSR (crow[n_owned+1], col, val[nnz]);
 *   block = 3: 3x3 block-CSR of a 3-dof operator (crow/col = node-level pattern of the n_owned/3 owned nodes, val = nnz
 *              row-major blocks); rows, halo lists and the boundary table are dof-level (3*node + component).
 * sym_host[P] = every rank's symmetric buffer as mapped in this process.  For neighbour k: nbr_host[k] = its rank,
 * send_idx[send_ptr_host[k]..send_ptr_host[k+1]) = my owned entries it needs, ghost_off_host[k] = index in ITS p where my
 * block starts.  One iteration = two kernels in a CUDA graph (merged-reduction loop): SpMV + three dot products, then one
 * vector pass; the halo exchange is peer stores + epoch flags, the all-reduce "LL" words (value and epoch in one 8-byte
 * store) -- there is no NCCL call in the loop.  Convergence is tested on the exactly summed r.r (r.z) one SpMV late, so the
 * returned state is the reference's at its break.  Rows [0,n_interior) must not reference ghost columns (their SpMV
 * overlaps the exchange); pass 0 if the rows are not ordered that way.  work = 2*n_owned. */
int femb_dist_cg_solve(int rank, int nranks, int64_t n_owned, int64_t n_interior, int64_t nnz, const int32_t* crow,
                       const int32_t* col, const double* val, const double* F, const uint8_t* mask, const double* minv,
                       double* u, double* work,
                       void* const* sym_host, int nnbr, const int32_t* nbr_host, const int32_t* send_ptr_host,
                       const int32_t* send_idx, const int64_t* ghost_off_host,
                       /* optional (NULL = separate push kernel): CSR over the boundary rows [n_interior,n_owned) of their
                        * destinations, bk = neighbour index, boff = offset in that neighbour's ghost block; lets the
                        * vector kernel store boundary values straight into the neighbours' ghost slots */
                       const int32_t* bptr, const uint8_t* bk, const int32_t* boff, double tol, int max_iter, double eps,
                       int check_every, int block, femb_cg_result* result_host, femb_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* FEMB200_H */
