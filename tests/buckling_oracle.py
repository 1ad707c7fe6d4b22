"""Numpy restatement of linear buckling (femb_solid_geometric, femb200/buckling.py, solver.buckling_modes) -- TEST INFRASTRUCTURE,
NOT PRODUCT CODE.

Geometric stiffness: at every point H[i,k] = du_k/dx_i = sum_a g_a[i] u_a[k], sigma = lam tr(H) I + mu (H + H^T),
s_ab = sum_q w_q |detJ_q| g_a^T sigma_q g_b, element matrix = s (x) I3.  `column` builds the Kuhn-split cantilever column of the
tests; `dense_case` solves the reference state with a sparse direct solve and returns the dense reduced pencil (K_G_ff, K_ff).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl
import scipy.sparse as sp
import scipy.sparse.linalg as sla

from oracle import fem_oracle as O
from oracle import modes_oracle as MO

KUHN = ((0, 1, 2, 6), (0, 2, 3, 6), (0, 3, 7, 6), (0, 7, 4, 6), (0, 4, 5, 6), (0, 5, 1, 6))
HEX_OFF = ((0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1))


def lame(E, nu):
    c = E / ((1 + nu) * (1 - 2 * nu))
    return c * nu, c * (1 - 2 * nu) / 2


# ------------------------------------------------------------------------------------------------------------------ rules

def rule14():
    """The degree-5 14-point tet rule of femb_mass_points(C3D10): [14, 4] rows (xi, eta, zeta, w), weights summing to 1/6."""
    a, wa = (0.3108859192633006098, 0.09273525031089122640), (0.01878132095300264180, 0.01224884051939365826)
    b, wb = 0.04550370412564964949, 0.007091003462846911073
    rows = []
    for o in range(2):
        c = 1 - 3 * a[o]
        rows += [[a[o], a[o], a[o], wa[o]], [c, a[o], a[o], wa[o]], [a[o], c, a[o], wa[o]], [a[o], a[o], c, wa[o]]]
    h = 0.5 - b
    rows += [[p[0], p[1], p[2], wb] for p in ((b, b, h), (b, h, b), (h, b, b), (b, h, h), (h, b, h), (h, h, b))]
    return np.array(rows)


def collapsed_gauss(n):
    """Conical-product rule on the unit tet: n-point Gauss-Legendre on the cube mapped by xi = u, eta = v (1-u),
    zeta = w (1-u)(1-v) (Jacobian (1-u)^2 (1-v)); exact for polynomials of degree <= 2n - 3."""
    x, w = np.polynomial.legendre.leggauss(n)
    x, w = (x + 1) / 2, w / 2
    rows = []
    for u, wu in zip(x, w):
        for v, wv in zip(x, w):
            for t, wt in zip(x, w):
                rows.append([u, v * (1 - u), t * (1 - u) * (1 - v), wu * wv * wt * (1 - u) ** 2 * (1 - v)])
    return np.array(rows)


# ------------------------------------------------------------------------------------------------------- element matrices

def _sigma(H, E, nu):
    lam, mu = lame(E, nu)
    tr = np.einsum("mii->m", H)
    return lam * tr[:, None, None] * np.eye(3) + mu * (H + np.transpose(H, (0, 2, 1)))


def _kron3(s):
    M, n = s.shape[:2]
    return np.einsum("mab,ij->maibj", s, np.eye(3)).reshape(M, 3 * n, 3 * n)


def c3d4_KG(coords, tets, u, E, nu):
    g = O.c3d4_gradients(coords, tets)                                   # [M, 4, 3]
    V = O.tet_volumes(coords, tets)
    H = np.einsum("mai,mak->mik", g, np.asarray(u, dtype=np.float64)[np.asarray(tets)])
    s = V[:, None, None] * np.einsum("mai,mij,mbj->mab", g, _sigma(H, E, nu), g)
    return _kron3(s)


def c3d10_KG(coords, tets, u, E, nu, points):
    u = np.asarray(u, dtype=np.float64)
    ue = u[np.asarray(tets)]
    s = 0.0
    for p in np.asarray(points, dtype=np.float64):
        g = O.shape_gradients("c3d10", coords, tets, p[:3])             # [M, 10, 3]
        det = np.abs(np.linalg.det(O.jacobian("c3d10", coords, tets, p[:3])))
        H = np.einsum("mai,mak->mik", g, ue)
        s = s + (p[3] * det)[:, None, None] * np.einsum("mai,mij,mbj->mab", g, _sigma(H, E, nu), g)
    return _kron3(s)


def c3d10_K(coords, tets, E, nu, points):
    return O.solid_K("c3d10", coords, tets, E, nu, points=points)


# ---------------------------------------------------------------------------------------------------------------- meshes

def column(k, L=20.0, quadratic=False, jitter=0.0, seed=0):
    """Cantilever column [0,1]^2 x [0,L] of k x k x (L k) hex cells, six Kuhn tets each; quadratic: C3D10 with local nodes 0 <-> 1
    swapped (detJ > 0 for the element's natural coordinates).  Returns (coords [N,3], elements)."""
    nz = int(round(L * k))
    ax = np.arange(k + 1) / k
    az = np.arange(nz + 1) / nz * L
    X, Y, Z = np.meshgrid(ax, ax, az, indexing="ij")
    c = np.stack([X, Y, Z], axis=-1).reshape(-1, 3)
    if jitter:
        inner = ((c[:, :2] > 0) & (c[:, :2] < 1)).all(axis=1) & (c[:, 2] > 0) & (c[:, 2] < L)
        c = c + np.random.default_rng(seed).uniform(-1, 1, c.shape) * inner[:, None] * (jitter / k)
    I, J, K = np.meshgrid(np.arange(k), np.arange(k), np.arange(nz), indexing="ij")
    hexes = np.stack([((I + a) * (k + 1) + (J + b)) * (nz + 1) + (K + d) for (a, b, d) in HEX_OFF], axis=-1).reshape(-1, 8)
    tets = hexes[:, np.array(KUHN)].reshape(-1, 4)
    if quadratic:
        c, t10 = O.c3d4_to_c3d10(c, tets[:, [1, 0, 2, 3]])
        return np.asarray(c), np.asarray(t10, dtype=np.int64)
    return c, tets


def clamp_base(c):
    return np.nonzero(np.abs(np.asarray(c)[:, 2]) < 1e-12)[0]


def top_load(c, total=-1.0):
    """F [N,3]: `total` in z shared equally by the nodes of the top face (z = max)."""
    c = np.asarray(c)
    top = np.abs(c[:, 2] - c[:, 2].max()) < 1e-12
    F = np.zeros_like(c)
    F[top, 2] = total / top.sum()
    return F


def euler(L=20.0, E=1.0):
    """pi^2 E I / (4 L^2) of the unit square section clamped at one end."""
    return np.pi ** 2 * E / 12.0 / (4 * L ** 2)


# ---------------------------------------------------------------------------------------------------------------- solves

def assemble(Ke, tets, N, pattern=None):
    pattern = pattern if pattern is not None else MO.node_pattern(tets, N)
    return MO.assemble_bsr3(Ke, tets, N, pattern)


def dense_case(coords, tets, F, fixed, E, nu, points=None):
    """Reference state and pencil: (u [N,3], K (scipy), KG (scipy), free bool [3N], pattern, kval, kgval)."""
    coords = np.asarray(coords, dtype=np.float64)
    N = coords.shape[0]
    pat = MO.node_pattern(tets, N)
    quad = np.asarray(tets).shape[1] == 10
    kval = assemble(c3d10_K(coords, tets, E, nu, points) if quad else O.c3d4_K(coords, tets, E, nu), tets, N, pat)
    K = MO.bsr_matrix(pat[0], pat[1], kval).tocsr()
    free = MO.dof_mask(N, fixed).astype(bool)
    u = np.zeros(3 * N)
    u[free] = sla.spsolve(K[free][:, free].tocsc(), np.asarray(F, dtype=np.float64).reshape(-1)[free])
    u = u.reshape(N, 3)
    kgval = assemble(c3d10_KG(coords, tets, u, E, nu, points) if quad else c3d4_KG(coords, tets, u, E, nu), tets, N, pat)
    KG = MO.bsr_matrix(pat[0], pat[1], kgval).tocsr()
    return u, K, KG, free, pat, kval, kgval


def lowest_load_factors(K, KG, free, k=4):
    """The k lowest positive load factors of (K + lam K_G) phi = 0 on the free dofs (dense for small models, Lanczos otherwise)."""
    Kf, Gf = K[free][:, free], KG[free][:, free]
    if Kf.shape[0] <= 3000:
        nu = sl.eigh(Gf.toarray(), Kf.toarray(), eigvals_only=True, subset_by_index=[0, k - 1])
    else:
        nu = np.sort(sla.eigsh(Gf.tocsc(), k=k, M=Kf.tocsc(), which="SA", tol=1e-12)[0])
    return np.where(nu < 0, -1.0 / np.where(nu < 0, nu, -1.0), np.inf)


class PencilBackend(MO.NumpyBackend):
    """MO.NumpyBackend of (A, B) = (K_G, K) with the Jacobi preconditioner of B (buckling.JacobiBackend)."""

    def __init__(self, brow, bcol, kgval, kval, mask):
        super().__init__(brow, bcol, kgval, kval, mask)
        d = self.M.diagonal()
        self.dinv = np.where((self.mask != 0) & (d != 0), 1.0 / np.where(d != 0, d, 1.0), 0.0)
