"""Linear buckling on the GPU: femb_solid_geometric against its numpy restatement (tests/buckling_oracle.py), buckling_modes against
the dense pencil of the restatement, subdivided_buckling_modes against buckling_modes on the same finest mesh, and the error cases."""
import os
import sys

import numpy as np
import pytest
import torch

import buckling_oracle as B
from conftest import PKG

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(PKG, "solver"))

DEV = "cuda:0"
E, NU = 1.0, 0.3


@pytest.fixture(scope="module")
def env():
    import element
    import solver
    return element, solver


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def kg_device(el, quadratic, c, t, u, dtype, points=None):
    if quadratic:
        return el.compute_c3d10_KG_matrix(c, t, u, E, NU, integral_point=points, device=DEV, dtype=dtype)
    return el.compute_c3d4_KG_matrix(c, t, u, E, NU, device=DEV, dtype=dtype)


@pytest.mark.parametrize("quadratic", [False, True], ids=["c3d4", "c3d10"])
def test_kernel_matches_restatement(env, quadratic):
    el, _ = env
    c, t = B.column(3, L=1.0, quadratic=quadratic, jitter=0.3, seed=11)
    u = np.random.default_rng(5).standard_normal(c.shape)
    ref = B.c3d10_KG(c, t, u, E, NU, B.rule14()) if quadratic else B.c3d4_KG(c, t, u, E, NU)
    ct, tt, ut = torch.from_numpy(c), torch.from_numpy(t), torch.from_numpy(u)
    K64 = kg_device(el, quadratic, ct, tt, ut, torch.float64)
    assert rel(K64.cpu(), ref) <= 1e-12
    assert torch.equal(K64, K64.transpose(1, 2))                                              # bitwise symmetric
    assert torch.equal(K64, kg_device(el, quadratic, ct, tt, ut, torch.float64))             # repeated launch bit-identical
    assert torch.equal(K64, kg_device(el, quadratic, ct, tt.to(torch.int32), ut, torch.float64))   # int32 connectivity
    # fp32: coordinates and displacements are rounded to fp32 first, so the reference is the restatement on the rounded inputs
    c32, u32 = c.astype(np.float32).astype(np.float64), u.astype(np.float32).astype(np.float64)
    ref32 = B.c3d10_KG(c32, t, u32, E, NU, B.rule14()) if quadratic else B.c3d4_KG(c32, t, u32, E, NU)
    for udt in (torch.float32, torch.float64):
        K32 = kg_device(el, quadratic, ct, tt, ut.to(udt), torch.float32)
        assert K32.dtype == torch.float32 and torch.equal(K32, K32.transpose(1, 2))
        assert rel(K32.cpu(), ref32) <= 1e-6, udt
    if quadratic:                                                                             # a caller's rule: 4-point Gauss collapsed
        pts = torch.from_numpy(B.collapsed_gauss(2))
        assert rel(kg_device(el, True, ct, tt, ut, torch.float64, pts).cpu(), B.c3d10_KG(c, t, u, E, NU, B.collapsed_gauss(2))) <= 1e-12


def case(quadratic, k=1, L=6.0):
    c, t = B.column(k, L, quadratic)
    F, fixed = B.top_load(c), B.clamp_base(c)
    return c, t, F, fixed, B.dense_case(c, t, F, fixed, E, NU, B.rule14() if quadratic else None)


@pytest.mark.parametrize("quadratic", [False, True], ids=["c3d4", "c3d10"])
def test_buckling_modes_match_dense_pencil(env, quadratic):
    _, sv = env
    c, t, F, fixed, (u, K, KG, free, *_) = case(quadratic)
    lam, X, ur, info = sv.buckling_modes(c, t, F, fixed, E, NU, num_eigs=4, tol=1e-10, return_info=True, verbose=False)
    assert info["status"] == "converged" and "freq_hz" not in info and info["static_iterations"] > 0
    ref = B.lowest_load_factors(K, KG, free, 4)
    assert np.abs(lam.cpu().numpy() / ref - 1).max() <= 1e-7
    assert rel(ur.cpu(), u) <= 1e-6                  # static_tol 1e-10 on the residual, cond(K_ff) ~ 1e4
    Xh = X.cpu().numpy()
    assert np.abs(Xh[~free]).max() == 0.0
    assert np.abs(Xh.T @ (K @ Xh) - np.eye(4)).max() <= 1e-10
    # (K + lam K_G) phi = -lam (K_G - nu K) phi: the convergence test bounds it by tol (lam |K_G|_1 + |K|_1) |phi|
    lh = lam.cpu().numpy()
    nK, nG = abs(K).sum(axis=1).max(), abs(KG).sum(axis=1).max()
    for j in range(4):
        r = K @ Xh[:, j] + lh[j] * (KG @ Xh[:, j])
        assert np.linalg.norm(r[free]) <= 10 * 1e-10 * (lh[j] * nG + nK) * np.linalg.norm(Xh[:, j])


def test_buckling_modes_repeat_bitwise_and_fp32(env):
    _, sv = env
    c, t, F, fixed, _ = case(False)
    a = sv.buckling_modes(c, t, F, fixed, E, NU, num_eigs=3, verbose=False)
    b = sv.buckling_modes(c, t, F, fixed, E, NU, num_eigs=3, verbose=False)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    f = sv.buckling_modes(c, t, F, fixed, E, NU, num_eigs=3, dtype=torch.float32, verbose=False)
    assert all(x.dtype == torch.float32 for x in f)
    assert rel(f[0].cpu(), a[0].cpu()) <= 1e-6


def clamp_base_t(c):
    return torch.nonzero(c[:, 2].abs() < 1e-12).reshape(-1)


def top_load_t(c, t):
    return torch.from_numpy(B.top_load(c.cpu().numpy())).to(c.device)


def test_subdivided_matches_buckling_modes_and_tracks_euler(env):
    _, sv = env
    c, t = B.column(1)
    res = {}
    for levels in (0, 1, 2):
        lam, X, u, cf, tf, info = sv.subdivided_buckling_modes(c, t, levels, top_load_t, clamp_base_t, E, NU, num_eigs=2, tol=1e-10,
                                                               return_info=True, verbose=False)
        assert info["status"] == "converged" and len(info["levels"]) == levels + 1
        res[levels] = (lam, cf, tf, info)
    lam, cf, tf, info = res[1]
    lj, Xj, uj, ij = sv.buckling_modes(cf, tf, top_load_t(cf, tf), clamp_base_t(cf), E, NU, num_eigs=2, tol=1e-10, max_iter=20000,
                                       return_info=True, verbose=False)
    assert ij["status"] == "converged"
    assert np.abs(lam.cpu().numpy() / lj.cpu().numpy() - 1).max() <= 1e-7
    assert 5 * info["iterations"] <= ij["iterations"], (info["iterations"], ij["iterations"])   # 5,784 Jacobi iterations in numpy
    assert info["static_iterations"] < ij["static_iterations"]
    # the C3D4 column's locking error falls like h^2 toward Euler's load: lam_1 / Euler of the numpy restatement on these meshes
    ratio = [float(res[k][0][0]) / B.euler() for k in (0, 1, 2)]
    assert np.abs(np.array(ratio) / [3.6260, 1.5603, 1.2043] - 1).max() <= 1e-3, ratio


def test_error_cases(env):
    _, sv = env
    c, t, F, fixed, _ = case(False)
    with pytest.raises(ValueError, match=r"\[M,4\]"):
        sv.buckling_modes(c, np.zeros((3, 8), dtype=np.int64), F, fixed, E, NU, verbose=False)
    for k in (0, 13):
        with pytest.raises(ValueError, match="num_eigs"):
            sv.buckling_modes(c, t, F, fixed, E, NU, num_eigs=k, verbose=False)
    with pytest.raises(ValueError, match="zero"):
        sv.buckling_modes(c, t, np.zeros_like(F), fixed, E, NU, verbose=False)
    with pytest.raises(ValueError, match="free-free"):
        sv.buckling_modes(c, t, F, [], E, NU, verbose=False)
    with pytest.raises(ValueError, match="did not converge: relative residual"):
        sv.buckling_modes(c, t, F, fixed, E, NU, static_max_iter=3, verbose=False)
    with pytest.raises(ValueError, match="did not converge: relative residual"):   # one node clamped: rigid rotations remain
        sv.buckling_modes(c, t, F, fixed[:1], E, NU, static_max_iter=2000, verbose=False)
    c10, t10 = B.column(1, 6.0, quadratic=True)
    with pytest.raises(ValueError, match=r"\[M,4\]"):
        sv.subdivided_buckling_modes(c10, t10, 1, top_load_t, clamp_base_t, E, NU, verbose=False)
    with pytest.raises(ValueError, match="did not converge"):
        sv.subdivided_buckling_modes(c, t, 1, top_load_t, clamp_base_t, E, NU, static_max_iter=1, verbose=False)


def test_tension_gives_no_buckling(env):
    """Uniform uniaxial tension: Poisson 0, so the clamp adds no lateral stress, and F = K u for u = (0, 0, z) -- the consistent
    nodal loads of a uniform traction on the top face.  K_G is positive definite on the free dofs: every nu > 0, every lam = inf."""
    _, sv = env
    c, t = B.column(1, 6.0)
    fixed = B.clamp_base(c)
    _, K, _, free, *_ = B.dense_case(c, t, B.top_load(c), fixed, E, 0.0)
    F = (K @ np.stack([0 * c[:, 0], 0 * c[:, 0], c[:, 2]], axis=1).reshape(-1)) * free
    lam, X, u, info = sv.buckling_modes(c, t, F.reshape(-1, 3), fixed, E, 0.0, num_eigs=3, max_iter=300, return_info=True,
                                        verbose=False)
    assert np.all(info["nu"] > 0) and torch.isinf(lam).all()
