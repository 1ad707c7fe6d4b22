"""Linear buckling without a GPU: the numpy restatement of the geometric stiffness (tests/buckling_oracle.py) -- its invariants, a
patch test and the C3D10 rule --, the LOBPCG driver (femb200/modes.py) on the (K_G, K) pencil with the Jacobi and the multigrid
preconditioner, convergence of the column's load factor to Euler's, and argument validation of femb_solid_geometric."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sl

import buckling_oracle as B
import mg_oracle as G
from femb200 import buckling, modes
from oracle import modes_oracle as MO

E, NU = 1.0, 0.3


def jittered(quadratic, seed=3):
    """A short jittered column: straight-sided elements, every node but the outer boundary moved."""
    return B.column(2, L=2.0, quadratic=quadratic, jitter=0.25, seed=seed)


def kg_of(quadratic, c, t, u, points=None):
    return B.c3d10_KG(c, t, u, E, NU, B.rule14() if points is None else points) if quadratic else B.c3d4_KG(c, t, u, E, NU)


@pytest.mark.parametrize("quadratic", [False, True], ids=["c3d4", "c3d10"])
def test_geometric_stiffness_invariants(quadratic):
    c, t = jittered(quadratic)
    rng = np.random.default_rng(1)
    u1, u2 = rng.standard_normal(c.shape), rng.standard_normal(c.shape)
    K1, K2, K12 = kg_of(quadratic, c, t, u1), kg_of(quadratic, c, t, u2), kg_of(quadratic, c, t, 2.0 * u1 - 3.0 * u2)
    scale = np.abs(K1).max()
    assert np.abs(K1 - np.transpose(K1, (0, 2, 1))).max() <= 1e-14 * scale                 # symmetric
    nen = t.shape[1]
    for d in range(3):                                                                       # translations in the null space
        e = np.zeros(3 * nen)
        e[d::3] = 1.0
        assert np.abs(K1 @ e).max() <= 1e-13 * scale
    assert np.abs(K12 - (2.0 * K1 - 3.0 * K2)).max() <= 1e-13 * np.abs(K12).max()         # linear in u


@pytest.mark.parametrize("quadratic", [False, True], ids=["c3d4", "c3d10"])
def test_patch_uniaxial_stress(quadratic):
    """u affine with stress s e_z (x) e_z: v^T K_G v = s V sum_i (dv_i/dz)^2 for every affine v."""
    c, t = jittered(quadratic, seed=5)
    s = 0.7
    u = np.stack([-NU * s / E * c[:, 0], -NU * s / E * c[:, 1], s / E * c[:, 2]], axis=1)
    KG = B.assemble(kg_of(quadratic, c, t, u), t, c.shape[0])
    Kg = MO.bsr_matrix(*MO.node_pattern(t, c.shape[0]), KG).tocsr()
    V = 1.0 * 1.0 * 2.0
    rng = np.random.default_rng(2)
    for _ in range(3):
        A, b = rng.standard_normal((3, 3)), rng.standard_normal(3)
        v = (c @ A.T + b).reshape(-1)
        expect = s * V * np.sum(A[:, 2] ** 2)
        assert abs(v @ (Kg @ v) - expect) <= 1e-12 * abs(expect)


def test_rule14_matches_library_and_collapsed_gauss():
    from femb200 import ops
    assert np.array_equal(np.array(ops.mass_points(ops.C3D10)), B.rule14())
    assert abs(B.rule14()[:, 3].sum() - 1 / 6) < 1e-16 and abs(B.collapsed_gauss(4)[:, 3].sum() - 1 / 6) < 1e-16
    c, t = jittered(True, seed=7)
    u = np.random.default_rng(4).standard_normal(c.shape)
    K14, Kg = B.c3d10_KG(c, t, u, E, NU, B.rule14()), B.c3d10_KG(c, t, u, E, NU, B.collapsed_gauss(4))
    assert np.abs(K14 - Kg).max() <= 1e-13 * np.abs(Kg).max()


def test_load_factor_convention():
    assert np.array_equal(buckling.load_factors([-4.0, -0.5, 0.0, 2.0]), [0.25, 2.0, np.inf, np.inf])


def column_pencil(k=1, L=20.0, quadratic=False):
    c, t = B.column(k, L, quadratic)
    fixed = B.clamp_base(c)
    u, K, KG, free, pat, kval, kgval = B.dense_case(c, t, B.top_load(c), fixed, E, NU, B.rule14() if quadratic else None)
    return c, t, u, K, KG, free, pat, kval, kgval, MO.dof_mask(c.shape[0], fixed)


def test_lobpcg_on_the_pencil_matches_dense_eigh():
    c, t, u, K, KG, free, pat, kval, kgval, mask = column_pencil(1)
    be = B.PencilBackend(pat[0], pat[1], kgval, kval, mask)
    lam, X, info = buckling.solve(be, 4, tol=1e-10, max_iter=3000)
    assert info["status"] == "converged"
    ex = sl.eigh(KG[free][:, free].toarray(), K[free][:, free].toarray(), eigvals_only=True)
    assert np.abs(info["nu"] - ex[:4]).max() <= 1e-8 * np.abs(ex[0])
    assert np.all(np.diff(lam) >= 0) and np.abs(lam - (-1.0 / ex[:4])).max() <= 1e-8 * lam[0]
    assert np.abs(X[~free]).max() == 0.0 and np.abs(X.T @ (K @ X) - np.eye(4)).max() < 1e-10


# Lowest load factor over Euler's for the k x k x 20k column (unit square section, L = 20, clamped base, unit compression shared by
# the top-face nodes).  C3D4 locks in bending: the error is O(h^2) and Richardson extrapolation of k = 4 and 8 lands on Euler.
C3D4_COLUMN = {1: 3.63, 2: 1.68, 3: 1.31, 4: 1.18, 6: 1.080, 8: 1.045}


def test_c3d4_column_converges_to_euler():
    ratio = {}
    for k in C3D4_COLUMN:
        c, t, u, K, KG, free, *_ = column_pencil(k)
        ratio[k] = B.lowest_load_factors(K, KG, free, 2)[0] / B.euler()
    for k, r in C3D4_COLUMN.items():
        assert abs(ratio[k] - r) <= 0.006 * r, (k, ratio[k], r)
    assert abs((4 * ratio[8] - ratio[4]) / 3 - 1.0) <= 0.01, ratio


def test_c3d10_column_close_to_euler():
    c, t, u, K, KG, free, *_ = column_pencil(2, quadratic=True)
    r = B.lowest_load_factors(K, KG, free, 2)[0] / B.euler()
    assert abs(r - 1.0) <= 0.005, r          # 1.0016 measured with this restatement


@pytest.fixture(scope="module")
def column_levels():
    """The 1 x 1 x 20 column refined 1, 2 and 3 times: hierarchy, finest K and K_G (reference state from a direct solve)."""
    c, t = B.column(1)
    out = {}
    for L in (1, 2, 3):
        levels, kval, mval, cf, tf = G.numpy_hierarchy(c, t, L, B.clamp_base, E, NU, 1.0)
        u, K, KG, free, pat, kval2, kgval = B.dense_case(cf, tf, B.top_load(cf), B.clamp_base(cf), E, NU)
        assert np.array_equal(kval, kval2)
        out[L] = (levels, kval, kgval, K, KG, free)
    return out


def test_multigrid_iterations_flat_and_far_below_jacobi(column_levels):
    its = {}
    for L, (levels, kval, kgval, K, KG, free) in column_levels.items():
        nu, S, info = modes.lobpcg(G.NumpyMultilevelBackend(levels, kgval, kval), 4, tol=1e-8, max_iter=300)
        assert info["status"] == "converged", L
        its[L] = info["iterations"]
        if L == 3:
            ref = B.lowest_load_factors(K, KG, free, 4)
            assert np.abs(buckling.load_factors(nu) / ref - 1).max() <= 1e-6        # tol 1e-8 on the backward error: 2.5e-7 seen
            top = levels[-1]
            # Jacobi on the same 38,880 free dofs: not converged after 20x the multigrid count (a complete Jacobi run takes over
            # 20,000 iterations here)
            nj, _, ij = modes.lobpcg(B.PencilBackend(top["brow"], top["bcol"], kgval, kval, top["mask"]), 4, tol=1e-8, max_iter=20 * its[3])
            print(f"multigrid iterations {its}; Jacobi at 3 levels after {ij['iterations']}: {ij['status']}")
            assert ij["status"] == "maxiter"
    assert max(its.values()) - min(its.values()) <= 4 and its[3] <= its[1] + 4, its


def test_geometric_entry_validates_arguments_without_gpu():
    from femb200 import _lib
    L = _lib.lib
    buf = (ctypes.c_double * 64)()
    p = ctypes.addressof(buf)
    pts = (ctypes.c_double * 68)(*[0.25] * 68)

    def err(rc, word):
        assert rc == 1 and word in L.femb_last_error(), L.femb_last_error()

    # femb_solid_geometric(kind, coords, fp, conn, ib, M, disp, pts_host, nq, E, nu, out, stream)
    err(L.femb_solid_geometric(8, p, 8, p, 8, 1, p, pts, 1, 1.0, 0.3, p, None), b"C3D4 or C3D10")
    err(L.femb_solid_geometric(6, p, 8, p, 8, 1, p, pts, 1, 1.0, 0.3, p, None), b"C3D4 or C3D10")
    err(L.femb_solid_geometric(4, p, 2, p, 8, 1, p, None, 0, 1.0, 0.3, p, None), b"fp in {4,8}")
    err(L.femb_solid_geometric(4, p, 8, p, 3, 1, p, None, 0, 1.0, 0.3, p, None), b"ib in {4,8}")
    err(L.femb_solid_geometric(4, p, 8, p, 8, -1, p, None, 0, 1.0, 0.3, p, None), b"M >= 0")
    err(L.femb_solid_geometric(10, p, 8, p, 8, 1, p, None, 14, 1.0, 0.3, p, None), b"pts_host")
    err(L.femb_solid_geometric(10, p, 8, p, 8, 1, p, pts, 0, 1.0, 0.3, p, None), b"nq <= 16")
    err(L.femb_solid_geometric(10, p, 8, p, 8, 1, p, pts, 17, 1.0, 0.3, p, None), b"nq <= 16")
    err(L.femb_solid_geometric(4, p, 8, p, 8, 1, None, None, 0, 1.0, 0.3, p, None), b"non-null")
    err(L.femb_solid_geometric(10, p, 8, p, 8, 1, p, pts, 14, 1.0, 0.3, None, None), b"non-null")
    assert L.femb_solid_geometric(4, None, 8, None, 8, 0, None, None, 0, 1.0, 0.3, None, None) == 0   # empty: no launch
