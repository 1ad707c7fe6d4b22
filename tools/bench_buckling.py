#!/usr/bin/env python
"""Linear buckling on one B200: the geometric-stiffness kernel femb_solid_geometric against its byte model, and time to solution of
subdivided_buckling_modes (multigrid) against buckling_modes (Jacobi) on the same finest column mesh.  Writes one JSON (card name,
power limit and max SM clock read in the same run).

    python tools/bench_buckling.py [--k 2] [--levels 3] [--out results.json]

The JSON is also printed on stdout; without --out it is written to the system temporary directory.

Kernel workloads: BASELINE config 2 (kuhn_cube(69) as C3D10, 1,971,054 elements, default 14-point rule) and the finest mesh of
config 5 (kuhn_cube(8) refined 3 times, 1,572,864 C3D4), fp64, displacement = a smooth field.  Byte model (algorithmic): C3D4
M (4 ib + 1152) + 48 N (connectivity, the [12,12] output, coordinates and displacements once); C3D10 M (10 ib + 7200) + 48 N.  The
HBM peak is measured in the same run with a 4 GB device-to-device copy.  Outputs are larger than the 126 MB L2.

Time to solution: the k x k x 20k column (L = 20, clamped base, unit compression on the top face) refined 1 .. `levels` times, both
solvers on each finest mesh, 4 pairs, tol 1e-8; the reference static solve is part of each call.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "cuda-powered-mesh-handling-and-iterative-solvers_b200")
for p in (ROOT, PKG, os.path.join(PKG, "solver"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import buckling_oracle as B  # noqa: E402
import element as el  # noqa: E402
import solver as sv  # noqa: E402
from femb200 import buckling, hybrid, meshgen, modes, multigrid  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--k", type=int, default=2)
ap.add_argument("--levels", type=int, default=3)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--jacobi-max-iter", type=int, default=40000)
ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "bench_buckling.json"))
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_buckling.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
out = {"card": card}
E, NU, TOL, NEIG = 1.0, 0.3, 1e-8, 4


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


# ---------------------------------------------------------------- measured HBM peak (device-to-device copy, 2 x 4 GB moved)
src = torch.empty(2 ** 29, device=dev, dtype=torch.float64)
dst = torch.empty_like(src)
ms = events(lambda: dst.copy_(src), a.reps)
hbm = 2 * src.numel() * 8 / ms / 1e6
out["hbm_copy_GBps"] = round(hbm, 1)
del src, dst


# ---------------------------------------------------------------- femb_solid_geometric
def kernel_case(name, coords, conn, fn, bytes_model):
    N, M = coords.shape[0], conn.shape[0]
    u = torch.stack([torch.sin(coords[:, 2]), torch.cos(coords[:, 0]), coords[:, 1] * coords[:, 2]], dim=1).contiguous()
    res = {}
    buf = [None]

    def run():
        buf[0] = None          # release the previous output first: no cudaMalloc of a multi-GB block inside the timed region
        buf[0] = fn(coords, conn, u)

    ms = events(run, a.reps)
    b = bytes_model(M, N)
    res = {"elements": M, "nodes": N, "ms": round(ms, 3), "model_GB": round(b / 1e9, 3), "GBps": round(b / ms / 1e6, 1),
           "share_of_measured_hbm": round(b / ms / 1e6 / hbm, 3)}
    out[name] = res
    buf[0] = None
    torch.cuda.empty_cache()


c1, t1 = meshgen.kuhn_cube(69, device=dev)
c10, e10 = meshgen.p1_to_p2_lattice(69, meshgen.swap01(t1), device=dev)
del c1, t1
kernel_case("geometric_c3d10_config2", c10, e10,
            lambda c, t, u: el.compute_c3d10_KG_matrix(c, t, u, E, NU, device=dev, dtype=torch.float64),
            lambda M, N: M * (10 * 8 + 7200) + 48 * N)
del c10, e10
c4, t4 = meshgen.kuhn_cube(8, device=dev)
for _ in range(3):
    c4, t4, _p = hybrid.refine_once(c4, t4, el)
kernel_case("geometric_c3d4_config5", c4.contiguous(), t4.contiguous(),
            lambda c, t, u: el.compute_c3d4_KG_matrix(c, t, u, E, NU, device=dev, dtype=torch.float64),
            lambda M, N: M * (4 * 8 + 1152) + 48 * N)
del c4, t4
torch.cuda.empty_cache()

# ---------------------------------------------------------------- time to solution on the column
c0, t0 = (torch.from_numpy(x) for x in B.column(a.k))


def clamp(c):
    return torch.nonzero(c[:, 2].abs() < 1e-12).reshape(-1)


def load(c, t):
    return torch.from_numpy(B.top_load(c.cpu().numpy())).to(c.device)


sv.subdivided_buckling_modes(c0, t0, 1, load, clamp, E, NU, max_iter=3, verbose=False)      # warm-up (module load, library paths)
out["column"] = {"coarse": f"{a.k} x {a.k} x {20 * a.k} hex cells, 6 Kuhn tets each, L = 20", "num_eigs": NEIG, "tol": TOL,
                 "euler_load": B.euler(), "jacobi_max_iter": a.jacobi_max_iter}
out["by_levels"] = {}
for levels in range(1, a.levels + 1):
    (lam, X, u, cf, tf, info), wall_mg = timed(lambda: sv.subdivided_buckling_modes(c0, t0, levels, load, clamp, E, NU, num_eigs=NEIG,
                                                                                   tol=TOL, return_info=True, verbose=False))
    F, fx = load(cf, tf), clamp(cf)
    (lj, Xj, uj, ij), wall_j = timed(lambda: sv.buckling_modes(cf, tf, F, fx, E, NU, num_eigs=NEIG, tol=TOL, max_iter=a.jacobi_max_iter,
                                                              return_info=True, verbose=False))
    out["by_levels"][levels] = {
        "dofs": info["levels"][-1]["dofs"],
        "multigrid": {"status": info["status"], "iterations": info["iterations"], "static_iterations": info["static_iterations"],
                      "seconds_total": round(wall_mg, 3), "seconds_lobpcg_loop": round(info["loop_ms"] / 1e3, 3),
                      "load_factors": [float(v) for v in lam.cpu()], "lam1_over_euler": float(lam[0]) / B.euler()},
        "jacobi": {"status": ij["status"], "iterations": ij["iterations"], "static_iterations": ij["static_iterations"],
                   "seconds_total": round(wall_j, 3), "seconds_lobpcg_loop": round(ij["loop_ms"] / 1e3, 3),
                   "load_factors": [float(v) for v in lj.cpu()]},
        "max_rel_load_factor_diff": float(np.max(np.abs(lam.cpu().numpy() / lj.cpu().numpy() - 1))),
        "speedup_time_to_solution": round(wall_j / wall_mg, 2)}
    del X, Xj
    torch.cuda.empty_cache()
info = {"iterations": out["by_levels"][a.levels]["multigrid"]["iterations"]}


# ---------------------------------------------------------------- per-iteration split of the multigrid solve, and its static solve
class Timed(buckling.MultilevelBackend):
    """Sync-timed kernels: host clock around each call ending in a device synchronise; residual = residual kernel + V-cycle."""
    acc = {"spmm": 0.0, "gram": 0.0, "combine": 0.0, "residual_and_vcycle": 0.0}

    def _t(self, name, fn, *args, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(self, *args, **kw)
        torch.cuda.synchronize()
        self.acc[name] += (time.perf_counter() - t0) * 1e3

    def spmm(self, *a, **k): self._t("spmm", modes.DeviceBackend.spmm, *a, **k)       # noqa: E704
    def gram(self, *a, **k): self._t("gram", modes.DeviceBackend.gram, *a, **k)       # noqa: E704
    def combine(self, *a, **k): self._t("combine", modes.DeviceBackend.combine, *a, **k)  # noqa: E704
    def residual(self, *a, **k): self._t("residual_and_vcycle", multigrid.MultilevelBackend.residual, *a, **k)  # noqa: E704


H = multigrid.Hierarchy(c0, t0, a.levels, clamp, E, NU, None, 0.0, dev, el)
(ur, sits, sres), t_static = timed(lambda: buckling.static_multigrid(H, load(H.coords, H.tets), 1e-10, 500))
top = H.L[-1]
KGe = el.compute_c3d4_KG_matrix(H.coords, H.tets, ur.reshape(-1, 3), E, NU, device=dev, dtype=torch.float64)
brow, bcol = top.plan.pattern(1)
from femb200 import ops  # noqa: E402
KG = ops.Bsr3.from_csr_values(brow, bcol, top.plan.assemble(KGe, 3))
del KGe
be = Timed(H, KG)
_, S, ti = modes.lobpcg(be, NEIG, tol=TOL, max_iter=info["iterations"])
its = max(ti["iterations"], 1)
out["multigrid_ms_per_iteration"] = {k: round(v / its, 3) for k, v in be.acc.items()}   # includes the start block's SpMM, Grams, combines
out["multigrid_static_solve"] = {"iterations": sits, "seconds": round(t_static, 3), "relative_residual": sres}

os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
