#!/usr/bin/env python
"""LOBPCG modal solver (lowest_modes) on one B200: fused K+M block SpMM against the 2m single SpMVs the subspace-iteration solver
issues, the per-iteration cost split, and time to solution.  Writes one JSON (card name and power limit read in the same run).

    python tools/bench_modes.py [--n 69] [--cantilever-n 40] [--out results.json]

The JSON is also printed on stdout; without --out it is written to the system temporary directory.

SpMM: BASELINE config 2 (P2 tets, Kuhn n=69: ~2 M C3D10, ~76 M 3x3 blocks; K and M values together ~11 GB, far above the
126 MB L2, so every pass streams the matrices from HBM).  Bytes are an algorithmic model kept here: fused SpMM = (4 + 2*72) nnzb
+ x read once (8 n m) + both Y written (16 n m); one SpMV = (4 + 72) nnzb + 16 n.
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
from femb200 import meshgen, modes, ops  # noqa: E402
from femb200._lib import check, lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=69)
ap.add_argument("--cantilever-n", type=int, default=40)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "bench_modes.json"))
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_modes.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
out = {"card": card}


def events_ms(fn, reps):
    fn()
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


# ---------------------------------------------------------------- config 2 operators
c1, t1 = meshgen.kuhn_cube(a.n, device=dev)
coords, e10 = meshgen.p1_to_p2_lattice(a.n, meshgen.swap01(t1), device=dev)
del c1, t1
N = coords.shape[0]
plan = ops.CsrPlan(e10, N, dev)
brow, bcol = plan.pattern(1)


def bsr(Ke_fn):
    Ke = Ke_fn()
    vals = plan.assemble(Ke, 3)
    del Ke
    return ops.Bsr3.from_csr_values(brow, bcol, vals)


K = bsr(lambda: el.compute_c3d10_K_matrix(coords, e10, 1.0, 0.3, device=dev, dtype=torch.float64))
M = bsr(lambda: el.compute_c3d10_M_matrix(coords, e10, 2.5, device=dev, dtype=torch.float64))
torch.cuda.synchronize()
nb, nnzb, n = K.nb, K.nnzb, 3 * K.nb
out["config2"] = {"elements": e10.shape[0], "nodes": N, "dofs": n, "nnzb": nnzb, "matrix_GB_K_plus_M": round(2 * 76 * nnzb / 1e9, 2)}
stream = torch.cuda.current_stream(dev).cuda_stream
P = modes._p

spmm = {}
for m in (4, 8, 16):
    X = torch.randn(n, m, device=dev, dtype=torch.float64)
    YK, YM = torch.empty_like(X), torch.empty_like(X)

    def fused():
        check(lib.femb_spmm_bsr3(nb, nnzb, P(K.brow), P(K.bcol), P(K.bval), P(M.bval), None, m, P(X), m, P(YK), P(YM), m, stream))

    cols = X.t().contiguous()                     # the column-major layout of vectorized_modal_solver's MultiVec
    yk, ym = torch.empty_like(cols), torch.empty_like(cols)

    def loop():
        for j in range(m):
            check(lib.femb_spmv_bsr3(nb, nnzb, P(K.brow), P(K.bcol), P(K.bval), P(cols[j]), P(yk[j]), stream))
            check(lib.femb_spmv_bsr3(nb, nnzb, P(M.brow), P(M.bcol), P(M.bval), P(cols[j]), P(ym[j]), stream))

    t_f, t_l = events_ms(fused, a.reps), events_ms(loop, a.reps)
    err = max(float((YK.t() - yk).abs().max() / yk.abs().max()), float((YM.t() - ym).abs().max() / ym.abs().max()))
    b_f = (4 + 2 * 72) * nnzb + 8 * n * m + 16 * n * m
    b_l = 2 * m * ((4 + 72) * nnzb + 16 * n)
    spmm[m] = {"fused_ms": round(t_f, 3), "spmv_loop_ms": round(t_l, 3), "speedup": round(t_l / t_f, 2),
               "fused_model_GB": round(b_f / 1e9, 2), "fused_GBps": round(b_f / t_f / 1e6, 1),
               "loop_model_GB": round(b_l / 1e9, 2), "loop_GBps": round(b_l / t_l / 1e6, 1), "max_rel_diff": err}
    del X, YK, YM, cols, yk, ym
out["spmm_config2"] = spmm


# ---------------------------------------------------------------- per-iteration split on config 2 (num_eigs = 10, capped)
class Timed(modes.DeviceBackend):
    """Sync-timed kernels: host clock around each call ending in a device synchronise."""
    acc = {"spmm": 0.0, "gram": 0.0, "combine": 0.0, "residual": 0.0}

    def _t(self, name, fn, *args, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(self, *args, **kw)
        torch.cuda.synchronize()
        self.acc[name] += (time.perf_counter() - t0) * 1e3

    def spmm(self, *a, **k): self._t("spmm", modes.DeviceBackend.spmm, *a, **k)       # noqa: E704
    def gram(self, *a, **k): self._t("gram", modes.DeviceBackend.gram, *a, **k)       # noqa: E704
    def combine(self, *a, **k): self._t("combine", modes.DeviceBackend.combine, *a, **k)  # noqa: E704
    def residual(self, *a, **k): self._t("residual", modes.DeviceBackend.residual, *a, **k)  # noqa: E704


fixed = torch.nonzero(coords[:, 0] == 0).reshape(-1)
be = Timed(K, M, sv._dof_mask(N, 3, fixed, dev))
iters = 4
for v in be.acc:
    be.acc[v] = 0.0
lam, S, info = modes.lobpcg(be, 10, tol=1e-8, max_iter=iters)
per = {k: round(v / iters, 3) for k, v in be.acc.items()}   # includes the start block's SpMM, Grams and combines
out["lobpcg_config2_num_eigs10"] = {"iterations": info["iterations"], "loop_ms": round(info["loop_ms"], 1),
                                    "kernel_ms_per_iteration": per, "block_width": modes.block_width(10)}
del be, S, K, M, plan, coords, e10
torch.cuda.empty_cache()

# ---------------------------------------------------------------- time to solution: P1 cantilever, ~200 k dofs
c, t = meshgen.kuhn_cube(a.cantilever_n, device=dev)
Kl = el.compute_c3d4_K_matrix(c, t, 1.0, 0.3, device=dev, dtype=torch.float64)
Ml = el.compute_c3d4_M_matrix(c, t, 2.5, device=dev, dtype=torch.float64)
fixed = torch.nonzero(c[:, 0] == 0).reshape(-1)
sv.lowest_modes(Kl, Ml, t, fixed, c.shape[0], num_eigs=6, max_iter=2, verbose=False)   # warm-up (plan, module load)
torch.cuda.synchronize()
t0 = time.perf_counter()
lam, X, info = sv.lowest_modes(Kl, Ml, t, fixed, c.shape[0], num_eigs=6, tol=1e-8, return_info=True, verbose=False)
torch.cuda.synchronize()
wall = time.perf_counter() - t0
out["cantilever"] = {"mesh": f"kuhn_cube({a.cantilever_n}) C3D4, x=0 face fixed", "dofs": 3 * c.shape[0], "tol": 1e-8,
                     "status": info["status"], "iterations": info["iterations"], "restarts": info["restarts"],
                     "seconds_total": round(wall, 3), "seconds_loop": round(info["loop_ms"] / 1e3, 3),
                     "lam": [float(v) for v in lam.cpu()], "max_residual": float(np.max(info["residuals"]))}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
