"""amg_lowest_modes without a GPU: the numpy restatement of the smoothed-aggregation setup and cycle (tests/amg_oracle.py) -- the
aggregates, the tentative prolongator, the Galerkin hierarchy on a free-free K, the symmetry of the cycle, independence of where the
mesh is placed, LOBPCG iteration counts against Jacobi on cantilevers of C3D4, C3D10 and C3D8 meshes at several sizes -- and
argument validation of the new C ABI entries."""
import ctypes

import numpy as np
import pytest

import amg_oracle as A
import buckling_oracle as BO
from femb200 import meshgen, modes
from oracle import fem_oracle as O
from oracle import modes_oracle as MO

E, NU, RHO = 1.0, 0.3, 2.5


def kuhn(n, jitter=0.2):
    c, t = meshgen.kuhn_cube(n, jitter=jitter)
    c, t = c.numpy(), t.numpy()
    pat = MO.node_pattern(t, c.shape[0])
    return c, t, pat, MO.assemble_bsr3(O.c3d4_K(c, t, E, NU), t, c.shape[0], pat), MO.assemble_bsr3(O.c3d4_mass(c, t, RHO), t, c.shape[0], pat)


def clamp_x0(c):
    return np.nonzero(np.abs(c[:, 0]) < 1e-12)[0]


def test_aggregates_cover_connect_and_roots_are_far_apart():
    c, t, (brow, bcol), kval, _ = kuhn(8)
    N = c.shape[0]
    mask = MO.dof_mask(N, clamp_x0(c))
    agg, n = A.aggregate(brow, bcol, mask)
    incl = mask.reshape(N, 3).any(axis=1)
    assert np.all(agg[~incl] == -1) and np.all(agg[incl] >= 0) and set(agg[incl]) == set(range(n))
    G = A.pattern((brow, bcol, None), N).tocsr()
    import scipy.sparse.csgraph as cg
    for a in range(n):
        nodes = np.nonzero(agg == a)[0]
        ncomp, _ = cg.connected_components(G[nodes][:, nodes], directed=False)
        assert ncomp == 1, a
    # roots: the node of each aggregate a at rank a; no two within distance 2
    import scipy.sparse as sp
    _, roots = A.mis_roots(brow, bcol, mask)
    G2 = (G @ G).tocsr()
    assert roots.size == n and (G2[roots][:, roots].multiply(1 - sp.eye(n).toarray())).count_nonzero() == 0
    assert np.array_equal(agg, A.aggregate(brow, bcol, mask)[0])


def test_tentative_is_orthonormal_and_reproduces_the_near_nullspace():
    c, t, (brow, bcol), kval, _ = kuhn(8)
    N = c.shape[0]
    mask = MO.dof_mask(N, clamp_x0(c))
    agg, n = A.aggregate(brow, bcol, mask)
    Pt, Bc, mc, cc = A.tentative(agg, n, mask, c)
    P = A.dof(Pt, 2 * n).toarray()
    kept = mc.astype(bool)
    assert np.abs(P.T @ P - np.diag(kept.astype(float))).max() <= 1e-13
    # B_f: the global rigid-body modes, masked
    Bf = A.rigid_rows(c, np.zeros(3), 1.0) * mask[:, None]
    assert np.abs(P @ Bc - Bf).max() <= 1e-13 * np.abs(Bf).max()


def test_free_free_hierarchy_keeps_the_rigid_modes_and_the_cycle_is_symmetric():
    c, t, (brow, bcol), kval, mval = kuhn(10)
    N = c.shape[0]
    mask = np.ones(3 * N, dtype=np.uint8)
    with pytest.raises(ValueError, match="shift > 0"):
        A.NumpyAmg((brow, bcol, kval), mask, c, coarse_dofs=150)
    T, lv_mask, B, x = (brow, bcol, kval), mask, None, c
    for _ in range(2):   # Galerkin operators of K are symmetric and annihilate the carried near-nullspace
        nodes = len(T[0]) - 1
        agg, n = A.aggregate(T[0], T[1], lv_mask)
        Pt, Bc, mc, cc = A.tentative(agg, n, lv_mask, x, B)
        Ad = A.dof(T, nodes)
        dinv = A.jacobi(Ad, lv_mask)
        P = A.spgemm(A.smoother(T, lv_mask, dinv, 4 / (3 * A.spectral_radius(Ad, dinv))), Pt, nodes, 2 * n)
        T = A.spgemm(A.transpose(P, 2 * n), A.spgemm(T, P, nodes, 2 * n), nodes, 2 * n)
        Ac = A.dof(T, 2 * n)
        assert abs(Ac - Ac.T).max() <= 1e-14 * abs(Ac).max()
        assert np.abs(Ac @ Bc).max() <= 1e-10 * abs(Ac).max() * np.abs(Bc).max()
        assert np.abs(A.dof(Pt, 2 * n) @ Bc - (B if B is not None else A.rigid_rows(c, np.zeros(3), 1.0))).max() <= 1e-12 * np.abs(Bc).max()
        lv_mask, B, x = mc, Bc, cc
    be = A.NumpyAmgBackend(brow, bcol, kval, mval, mask, c, shift=1.0, coarse_dofs=150)
    assert len(be.H.levels) >= 3
    rng = np.random.default_rng(4)
    V, W = rng.standard_normal((3 * N, 3)), rng.standard_normal((3 * N, 3))
    a, b = W.T @ be.H.apply(V), V.T @ be.H.apply(W)
    assert np.abs(a - b.T).max() <= 1e-12 * np.abs(a).max()


def iterations(c, t, Ke, Me, coarse_dofs, fixed_fn=clamp_x0, num_eigs=6, jacobi=False):
    N = c.shape[0]
    pat = MO.node_pattern(t, N)
    kval, mval = MO.assemble_bsr3(Ke, t, N, pat), MO.assemble_bsr3(Me, t, N, pat)
    mask = MO.dof_mask(N, fixed_fn(c))
    be = MO.NumpyBackend(*pat, kval, mval, mask) if jacobi else A.NumpyAmgBackend(*pat, kval, mval, mask, c, coarse_dofs=coarse_dofs)
    lam, S, info = modes.lobpcg(be, num_eigs, tol=1e-8, max_iter=5000)
    assert info["status"] == "converged"
    return info["iterations"], lam


def c3d4_case(n):
    c, t = meshgen.kuhn_cube(n, jitter=0.2)
    c, t = c.numpy(), t.numpy()
    return c, t, O.c3d4_K(c, t, E, NU), O.c3d4_mass(c, t, RHO)


def c3d10_case(n):
    c, t = meshgen.tet10_cube(n, jitter=0.1)
    c, t = c.numpy(), t.numpy()
    return c, t, BO.c3d10_K(c, t, E, NU, BO.rule14()), O.solid_mass("c3d10", c, t, RHO)


def c3d8_case(n):
    c, h = meshgen.hex_cube(n, jitter=0.1)
    c, h = c.numpy(), h.numpy()
    return c, h, O.c3d8_K(c, h, E, NU), O.solid_mass("c3d8", c, h, RHO)


# (mesh, sizes): the count may grow by at most GROWTH from the smallest to the largest size and must be at least 5x below Jacobi's on
# the largest.  Measured (coarsening at 150 free dofs, tol 1e-8): C3D4 15 / 20 / 25 (Jacobi 269), C3D10 24 / 28 (Jacobi 216), C3D8
# 14 / 19 (Jacobi 121)
GROWTH = 1.7
CASES = {"c3d4": (c3d4_case, (6, 12, 18)), "c3d10": (c3d10_case, (3, 6)), "c3d8": (c3d8_case, (6, 12))}


@pytest.mark.parametrize("kind", list(CASES))
def test_iteration_counts_stay_flat_and_beat_jacobi(kind):
    make, sizes = CASES[kind]
    counts = {}
    for n in sizes:
        c, t, Ke, Me = make(n)
        counts[n], lam = iterations(c, t, Ke, Me, 150)
    its_j, lj = iterations(c, t, Ke, Me, 0, jacobi=True)
    assert counts[sizes[-1]] <= GROWTH * counts[sizes[0]], counts
    assert 5 * counts[sizes[-1]] <= its_j, (counts, its_j)
    assert np.abs(lam - lj).max() <= 1e-7 * lj.max()


def test_hierarchy_does_not_depend_on_where_the_mesh_is_placed():
    """Every level re-centres its aggregates' rotation columns: the same mesh moved far from the origin drops the same near-nullspace
    columns on every level and converges in the same number of iterations."""
    c, t, Ke, Me = c3d4_case(12)
    N = c.shape[0]
    pat = MO.node_pattern(t, N)
    kval, mval = MO.assemble_bsr3(Ke, t, N, pat), MO.assemble_bsr3(Me, t, N, pat)
    mask = MO.dof_mask(N, clamp_x0(c))
    near = A.NumpyAmgBackend(*pat, kval, mval, mask, c, coarse_dofs=150)
    far = A.NumpyAmgBackend(*pat, kval, mval, mask, c + np.array([3e6, -2e6, 1e6]), coarse_dofs=150)
    assert len(near.H.levels) == len(far.H.levels) >= 3
    for a, b in zip(near.H.levels, far.H.levels):
        assert np.array_equal(a["mask"], b["mask"])
    its = [modes.lobpcg(be, 6, tol=1e-8, max_iter=500)[2]["iterations"] for be in (near, far)]
    assert its[0] == its[1], its


def test_flat_refined_column():
    import mg_oracle as G
    c, t = BO.column(1)
    for _ in range(2):
        c, t, _ = G.refine_once(c, t)
    its, _ = iterations(c, t, O.c3d4_K(c, t, E, NU), O.c3d4_mass(c, t, RHO), 150, fixed_fn=BO.clamp_base)
    assert its <= 60, its


def test_amg_entry_points_validate_arguments_without_gpu():
    from femb200 import _lib
    L = _lib.lib
    buf = (ctypes.c_double * 8192)()
    p = ctypes.addressof(buf)
    q, r = p + 8 * 2048, p + 8 * 4096
    n = ctypes.c_int64()

    def err(rc, word):
        assert rc == 1 and word in L.femb_last_error(), L.femb_last_error()

    err(L.femb_amg_aggregate(-1, p, p, None, q, ctypes.byref(n), None), b"nb")
    err(L.femb_amg_aggregate(4, None, p, None, q, ctypes.byref(n), None), b"non-null")
    assert L.femb_amg_aggregate(0, p, p, None, q, ctypes.byref(n), None) == 0 and n.value == 0
    err(L.femb_amg_tentative(4, 5, p, None, q, None, 1e-10, r, r, r, r, r, r, None), b"n_agg")
    err(L.femb_amg_tentative(4, 2, p, None, None, q, 1e-10, r, r, r, r, r, r, None), b"coords")
    err(L.femb_amg_tentative(4, 2, p, None, q, None, 1.5, r, r, r, r, r, r, None), b"drop")
    err(L.femb_amg_tentative(4, 2, p, None, q, None, 1e-10, r, None, r, r, r, r, None), b"non-null")
    err(L.femb_amg_tentative(4, 2, p, None, q, None, 1e-10, r, r, r, r, r, None, None), b"coords_c")
    err(L.femb_bsr3_spgemm(4, p, p, None, p, p, None, q, None, None, None, None), b"symbolic")
    err(L.femb_bsr3_spgemm(4, p, p, None, p, p, None, q, r, r, None, None), b"numeric")
    err(L.femb_bsr3_spgemm(4, None, p, p, p, p, p, q, r, r, None, None), b"non-null")
    err(L.femb_bsr3_transpose(-1, 2, 2, p, p, p, q, q, q, None), b"n_rows")
    err(L.femb_bsr3_transpose(2, 2, 2, p, None, p, q, q, q, None), b"non-null")
    err(L.femb_mg_transfer_bsr3(2, 2, 2, p, p, p, None, 17, q, 17, 0, r, 17, None), b"m <= 16")
    err(L.femb_mg_transfer_bsr3(2, 2, 2, None, p, p, None, 4, q, 4, 0, r, 4, None), b"non-null")
    err(L.femb_mg_transfer_bsr3(2, 2, 2, p, p, p, None, 4, q, 3, 0, r, 4, None), b"ldx")
    err(L.femb_mg_transfer_bsr3(2, 2, 2, p, p, p, None, 4, q, 4, 2, r, 4, None), b"accumulate")
    err(L.femb_mg_transfer_bsr3(2, 2, 2, p, p, p, None, 4, q, 4, 0, q + 8 * 8, 4, None), b"overlaps")
    assert L.femb_mg_transfer_bsr3(0, 2, 0, p, p, p, None, 4, q, 4, 0, r, 4, None) == 0
