#!/usr/bin/env python
"""Algebraic-multigrid modal and buckling solvers (amg_lowest_modes, amg_buckling_modes) on one B200.  Writes one JSON line (card
name and power limit read in the same run):
  config5   BASELINE config 5 (kuhn_cube(8) refined 3 times, 823,875 dofs, z = 0 face clamped, 6 pairs, tol 1e-8), the refined mesh
            passed flat: AMG against the geometric V-cycle (subdivided_lowest_modes) and Jacobi LOBPCG (lowest_modes)
  config2   BASELINE config 2 (P2 Kuhn lattice n = 69: 1,971,054 C3D10, 8.06 M dofs, z = 0 face clamped): AMG time to solution,
            Jacobi capped at --jacobi-cap iterations and reported as capped
  column    the 2 x 2 x 40 buckling column (L = 20) refined 3 times (278,307 dofs) passed flat: amg_buckling_modes against
            subdivided_buckling_modes
Each AMG entry holds the setup split (aggregation, tentative, lambda, spgemm, factor).  For config 5 and config 2 a second, sync-timed
LOBPCG run (as in bench_subdivided_modes.py: host clock around each backend call, ended by a device synchronise) gives the
per-iteration split -- residual + V-cycle, SpMM, Grams, combines -- beside the byte model of one V-cycle on m columns:
  per non-dense level  4 smoothing passes over A (76 nnzb + 24 n m each; the first pre-smoothing step reads no matrix, one pass forms
                       the residual) + R and P (76 nnzb(P) + 24 (n + n_c) m each)

    python tools/bench_amg_modes.py [--skip-c2] [--jacobi-cap 2000] [--out results.json]
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
from femb200 import amg, meshgen, modes, multigrid, ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--skip-c2", action="store_true")
ap.add_argument("--skip-jacobi", action="store_true")
ap.add_argument("--jacobi-cap", type=int, default=2000)
ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "bench_amg_modes.json"))
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_amg_modes.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
out = {"card": card}
E, NU, RHO, TOL, NEIG = 1.0, 0.3, 2.5, 1e-8, 6
KW = dict(device=dev, dtype=torch.float64, return_info=True, verbose=False)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


def zfix(c):
    return torch.nonzero(c[:, 2].abs() < 1e-12).reshape(-1)


def amg_entry(info, wall):
    return {"wall_s": wall, "iterations": info["iterations"], "status": info["status"], "loop_ms": info.get("loop_ms"),
            "setup_ms": info["setup_ms"], "levels": info["levels"], "operator_complexity": info["operator_complexity"]}


class Timed(multigrid.MultilevelBackend):
    """Sync-timed backend calls; residual = residual kernel + V-cycle."""

    def __init__(self, H):
        super().__init__(H)
        self.acc = {"spmm": 0.0, "gram": 0.0, "combine": 0.0, "residual_and_vcycle": 0.0}

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


def vcycle_bytes(H, m):
    """Byte model of one V(2,2) cycle on m columns (the dense coarsest level not counted)."""
    b = 0
    for lv, cl in zip(H.L[1:], H.L[:-1]):
        b += 4 * (76 * lv.A.nnzb + 24 * lv.n * m) + 2 * (76 * lv.P.nnzb + 24 * (lv.n + cl.n) * m)
    return b


def iteration_split(coords, Kl, Ml, elements):
    """Per-iteration split of amg_lowest_modes' LOBPCG on the same operators (a separate, sync-timed run)."""
    N = coords.shape[0]
    plan = ops.CsrPlan(elements, N, dev)
    brow, bcol = plan.pattern(1)
    K = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Kl, 3))
    M = ops.Bsr3.from_csr_values(brow, bcol, plan.assemble(Ml, 3))
    H = amg.AmgHierarchy(K, multigrid.dof_mask(N, zfix(coords), dev), coords, K=K, M=M)
    be = Timed(H)
    _, S, ti = modes.lobpcg(be, NEIG, tol=TOL, max_iter=500)
    its = max(ti["iterations"], 1)
    m = modes.block_width(NEIG)
    return {"iterations": its, "ms_per_iteration": {k: round(v / its, 3) for k, v in be.acc.items()},   # includes the start block
            "vcycle_bytes_model": {"m": m, "bytes": vcycle_bytes(H, m), "P_nnzb": [lv.P.nnzb for lv in H.L[1:]]}}


# warm-up: module load, library paths
c, t = meshgen.kuhn_cube(6)
sv.amg_lowest_modes(c, el.compute_c3d4_K_matrix(c, t, E, NU, device=dev, dtype=torch.float64),
                    el.compute_c3d4_M_matrix(c, t, RHO, device=dev, dtype=torch.float64), t.to(dev), zfix(c), num_eigs=NEIG, **KW)

# ---------------------------------------------------------------------------------------------------------- config 5
c0, t0 = meshgen.kuhn_cube(8)
(lg, Xg, cf, tf, ig), wall_g = timed(lambda: sv.subdivided_lowest_modes(c0, t0, 3, zfix, E, NU, RHO, num_eigs=NEIG, tol=TOL, **KW))
Kl = el.compute_c3d4_K_matrix(cf, tf, E, NU, device=dev, dtype=torch.float64)
Ml = el.compute_c3d4_M_matrix(cf, tf, RHO, device=dev, dtype=torch.float64)
(la, Xa, ia), wall_a = timed(lambda: sv.amg_lowest_modes(cf, Kl, Ml, tf, zfix(cf), num_eigs=NEIG, tol=TOL, **KW))
c5 = {"dofs": 3 * cf.shape[0], "amg": amg_entry(ia, wall_a), "geometric": {"wall_s": wall_g, "iterations": ig["iterations"]},
      "max_rel_eig_diff_vs_geometric": float((la - lg).abs().max() / lg.abs().max()), "eigenvalues": la.cpu().tolist()}
if not a.skip_jacobi:
    (lj, Xj, ij), wall_j = timed(lambda: sv.lowest_modes(Kl, Ml, tf, zfix(cf), cf.shape[0], num_eigs=NEIG, tol=TOL, **KW))
    c5["jacobi"] = {"wall_s": wall_j, "iterations": ij["iterations"], "status": ij["status"]}
    c5["max_rel_eig_diff_vs_jacobi"] = float((la - lj).abs().max() / lj.abs().max())
c5["amg_split"] = iteration_split(cf, Kl, Ml, tf)
del Kl, Ml
out["config5"] = c5
print(json.dumps({"config5": c5}), file=sys.stderr)

# ----------------------------------------------------------------------------------------------------------- column
cc, tc = (torch.from_numpy(x) for x in B.column(2))


def load(c, t):
    return torch.from_numpy(B.top_load(c.cpu().numpy())).to(c.device)


(lm, Xm, um, cfc, tfc, im), wall_m = timed(lambda: sv.subdivided_buckling_modes(cc, tc, 3, load, zfix, E, NU, num_eigs=4, tol=TOL, **KW))
(lb, Xb, ub, ib), wall_b = timed(lambda: sv.amg_buckling_modes(cfc, tfc, load(cfc, tfc), zfix(cfc), E, NU, num_eigs=4, tol=TOL, **KW))
out["column"] = {"dofs": 3 * cfc.shape[0], "amg": dict(amg_entry(ib, wall_b), static_iterations=ib["static_iterations"]),
                 "geometric": {"wall_s": wall_m, "iterations": im["iterations"], "static_iterations": im["static_iterations"]},
                 "load_factors": lb.cpu().tolist(), "max_rel_load_factor_diff": float((lb / lm - 1).abs().max())}
print(json.dumps({"column": out["column"]}), file=sys.stderr)

# ---------------------------------------------------------------------------------------------------------- config 2
if not a.skip_c2:
    n = 69
    c1, t1 = meshgen.kuhn_cube(n, device=dev)
    c2, e2 = meshgen.p1_to_p2_lattice(n, meshgen.swap01(t1), device=dev)
    Kl = el.compute_c3d10_K_matrix(c2, e2, E, NU, device=dev, dtype=torch.float64)
    Ml = el.compute_c3d10_M_matrix(c2, e2, RHO, device=dev, dtype=torch.float64)
    (la, Xa, ia), wall_a = timed(lambda: sv.amg_lowest_modes(c2, Kl, Ml, e2, zfix(c2), num_eigs=NEIG, tol=TOL, max_iter=500, **KW))
    c2o = {"dofs": 3 * c2.shape[0], "elements": e2.shape[0], "amg": amg_entry(ia, wall_a), "eigenvalues": la.cpu().tolist()}
    c2o["amg_split"] = iteration_split(c2, Kl, Ml, e2)
    if not a.skip_jacobi:
        (lj, Xj, ij), wall_j = timed(lambda: sv.lowest_modes(Kl, Ml, e2, zfix(c2), c2.shape[0], num_eigs=NEIG, tol=TOL, max_iter=a.jacobi_cap, **KW))
        c2o["jacobi"] = {"wall_s": wall_j, "iterations": ij["iterations"], "status": ij["status"], "capped_at": a.jacobi_cap}
    out["config2"] = c2o

line = json.dumps(out)
with open(a.out, "w") as f:
    f.write(line + "\n")
print(line)
