#!/usr/bin/env python
"""Multigrid-preconditioned modal solver (subdivided_lowest_modes) on one B200 against Jacobi LOBPCG (lowest_modes) on the same
finest K and M, the per-iteration cost split of the multigrid solve, and the damped-Jacobi smoothing kernel's rate.  Writes one
JSON (card name and power limit read in the same run).

    python tools/bench_subdivided_modes.py [--n 8] [--levels 3] [--out results.json]

The JSON is also printed on stdout; without --out it is written to the system temporary directory.

Mesh: BASELINE config 5 -- kuhn_cube(8) refined 3 times (1,572,864 C3D4, 824 k dofs), z = 0 face clamped, 6 pairs, tol 1e-8.

Byte model (algorithmic, kept here): one smoothing step with an input iterate = (4 + 72) nnzb (block column index + 3x3 block)
+ 24 n m (R and X_in read, X_out written).  A V(2,2) cycle costs about 4 such passes over the finest A (the first pre-smoothing
step starts from x = 0 and reads no matrix; one pass forms the residual for the restriction) plus a 1/8 geometric tail for the
coarser levels -- about 2.4 x the bytes of the iteration's fused K+M SpMM ((4 + 2 * 72) nnzb + 24 n m).
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
for p in (ROOT, PKG, os.path.join(PKG, "solver")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import element as el  # noqa: E402
import solver as sv  # noqa: E402
from femb200 import meshgen, modes, multigrid  # noqa: E402
from femb200._lib import check, lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=8)
ap.add_argument("--levels", type=int, default=3)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "bench_subdivided_modes.json"))
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_subdivided_modes.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
out = {"card": card}
E, NU, RHO, TOL, NEIG = 1.0, 0.3, 2.5, 1e-8, 6


def fixed_fn(c):
    return torch.nonzero(c[:, 2].abs() < 1e-12).reshape(-1)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


c0, t0 = meshgen.kuhn_cube(a.n)
cw, tw = meshgen.kuhn_cube(4)
sv.subdivided_lowest_modes(cw, tw, 1, fixed_fn, E, NU, RHO, max_iter=3, verbose=False)      # warm-up (module load, library paths)

# ---------------------------------------------------------------- time to solution: multigrid
(lam, X, cf, tf, info), wall_mg = timed(lambda: sv.subdivided_lowest_modes(c0, t0, a.levels, fixed_fn, E, NU, RHO, num_eigs=NEIG, tol=TOL,
                                                                         return_info=True, verbose=False))
out["mesh"] = {"coarse": f"kuhn_cube({a.n})", "levels": info["levels"], "fixed": "z = 0 face", "num_eigs": NEIG, "tol": TOL}
out["multigrid"] = {"status": info["status"], "iterations": info["iterations"], "restarts": info["restarts"], "seconds_total": round(wall_mg, 3),
                    "seconds_loop": round(info["loop_ms"] / 1e3, 3), "lam": [float(v) for v in lam.cpu()],
                    "max_residual": float(np.max(info["residuals"])), "smooth": multigrid.SMOOTH, "omega": multigrid.OMEGA}

# ---------------------------------------------------------------- time to solution: Jacobi lowest_modes on the same finest K, M
Kl = el.compute_c3d4_K_matrix(cf, tf, E, NU, device=dev, dtype=torch.float64)
Ml = el.compute_c3d4_M_matrix(cf, tf, RHO, device=dev, dtype=torch.float64)
fx = fixed_fn(cf)
sv.lowest_modes(Kl, Ml, tf, fx, cf.shape[0], num_eigs=NEIG, max_iter=2, verbose=False)        # warm-up (plan)
(lj, Xj, ij), wall_j = timed(lambda: sv.lowest_modes(Kl, Ml, tf, fx, cf.shape[0], num_eigs=NEIG, tol=TOL, max_iter=20000, return_info=True,
                                                       verbose=False))
out["jacobi"] = {"status": ij["status"], "iterations": ij["iterations"], "restarts": ij["restarts"], "seconds_total": round(wall_j, 3),
                 "seconds_loop": round(ij["loop_ms"] / 1e3, 3), "lam": [float(v) for v in lj.cpu()]}
out["max_rel_lam_diff"] = float(np.max(np.abs(lam.cpu().numpy() - lj.cpu().numpy()) / lj.cpu().numpy().max()))
out["speedup_time_to_solution"] = round(wall_j / wall_mg, 2)
del Kl, Ml, Xj
torch.cuda.empty_cache()


# ---------------------------------------------------------------- per-iteration split of the multigrid solve
class Timed(multigrid.MultilevelBackend):
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


H = multigrid.Hierarchy(c0, t0, a.levels, fixed_fn, E, NU, RHO, 0.0, dev, el)
be = Timed(H)
_, S, ti = modes.lobpcg(be, NEIG, tol=TOL, max_iter=info["iterations"])
its = max(ti["iterations"], 1)
out["multigrid_ms_per_iteration"] = {k: round(v / its, 3) for k, v in be.acc.items()}   # includes the start block's SpMM, Grams, combines
del S

# ---------------------------------------------------------------- femb_mg_smooth_bsr3 on the finest A, event-timed
top = H.L[-1]
A = top.A
n, nnzb = top.n, A.nnzb
stream = torch.cuda.current_stream(dev).cuda_stream
P = modes._p
smooth = {}
for m in (4, 8, 16):
    Rb = torch.randn(n, m, device=dev, dtype=torch.float64)
    Xi, Xo = torch.randn(n, m, device=dev, dtype=torch.float64), torch.empty(n, m, device=dev, dtype=torch.float64)

    def step():
        check(lib.femb_mg_smooth_bsr3(A.nb, nnzb, P(A.brow), P(A.bcol), P(A.bval), P(top.mask), P(top.dinv), multigrid.OMEGA, m, P(Rb), m,
                                      P(Xi), m, P(Xo), m, None, 0, stream))

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.reps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.reps
    b = (4 + 72) * nnzb + 24 * n * m
    smooth[m] = {"ms": round(ms, 4), "model_MB": round(b / 1e6, 1), "GBps": round(b / ms / 1e6, 1)}
out["mg_smooth_bsr3_finest"] = {"nnzb": nnzb, "dofs": n, "matrix_MB": round(76 * nnzb / 1e6, 1), "by_m": smooth,
                                "note": "matrix smaller than the 126 MB L2 is partly served from there across repetitions"
                                if 76 * nnzb < 126e6 else "matrix larger than the 126 MB L2: streamed from HBM"}
b_spmm = (4 + 2 * 72) * nnzb + 24 * n * 8
b_v = 4 * ((4 + 72) * nnzb + 24 * n * 8) * 8 / 7
out["byte_model_m8"] = {"fused_spmm_MB": round(b_spmm / 1e6, 1), "vcycle_MB": round(b_v / 1e6, 1), "ratio": round(b_v / b_spmm, 2)}

os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
