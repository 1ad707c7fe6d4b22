#!/usr/bin/env python
"""Benchmark of the FEM hot path (BASELINE.json metric: assembled elems/s; CG iters/s with SpMV GB/s vs HBM peak).

Workload (config.workload): BASELINE config 4, "P1 tet Poisson 64M tets" -- the configuration the north-star targets are
quoted on: Kuhn cube n=220, 63,888,000 C3D4 tets, 10,793,861 nodes, CSR nnz 160,738,381, fp64.  It fits one B200.
A step = one CG iteration of the reference's projected CG (solver.py:144-229) on the assembled CSR operator.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--n 220] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = CG iterations/s with everything resident in HBM (device events around one
graph-captured loop of exactly K iterations), `e2e` = the same through the public solver API with the load vector in pinned host memory and the
solution read back to the host inside the timed region of every call (median of repeated calls; the first call of the
process is reported as `first_call_ms`).  `roofline` is for the dominant kernel (the CSR SpMV).
`assembly` reports the second half of the metric (assembled elems/s, fused coords->CSR values) with its own roofline.
`config2` (1 GPU only) reports BASELINE config 2 beside it: P2 elasticity element K, assembly, block-CSR SpMV, Jacobi-PCG.
`--impl reference` times the UNMODIFIED reference (baseline/_ref/solver, installed by __graft_entry__.build(); run by
baseline/ref_arm.py in a subprocess, torch CPU on all host threads) on a bounded sample of the same workload; the C
restatement under oracle/ is reported beside it as a labelled second baseline (`cpu_baseline.port`).
`--dump-outputs DIR` (1 GPU) writes what the timed paths returned in their last step as DIR/<name>.npy (float64): the CG
solution and final r.r, the solution of the last e2e call and the assembled CSR values.  Inputs are seeded, so two builds
run with the same arguments can be compared output for output.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "cuda-powered-mesh-handling-and-iterative-solvers_b200")
for p in (ROOT, PKG, os.path.join(PKG, "solver")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC, UNIT = "cg_iters_per_s", "iter/s"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return json.load(open(path)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(n, kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture, only for the workload size it was captured on."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        d = json.load(open(path))
        return d[kernel]["traffic_bytes"] if d.get("n") == n else None
    except (OSError, KeyError, ValueError):
        return None


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi sampler (20 ms period).  Started well before the timed region (nvidia-smi needs a second to come up on an
    8-GPU box) and stopped after it; the reported clock is the median over samples taken while the GPU was busy
    (utilization >= 50 %), i.e. under the load of the very kernels being timed."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,"
         "utilization.gpu")

    def __init__(self, index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.stop)     # an exception before stop() must not leave nvidia-smi running
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.p = None
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 9]
        os.unlink(self.f.name)
        out["samples_total"] = len(rows)

        def util(r):
            try:
                return float(r[9])
            except ValueError:
                return 0.0
        busy = [r for r in rows if util(r) >= 50.0]
        rows = busy or rows
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows)
        out["sm_mhz"] = sm[len(sm) // 2]
        out["sm_max_mhz"] = float(rows[0][2])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out["reasons"] = [n for k, n in enumerate(names) if any("Active" in r[5 + k] and "Not" not in r[5 + k] for r in rows)]
        out["samples"] = len(rows)
        return out


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_SAMPLE = 1 << 21      # entries kept of a larger output (16 MB in float64), so that a dump stays well under 64 MB


def dump_sample(t):
    """`t` flattened to a float64 host array; an output of more than DUMP_SAMPLE entries is cut to a fixed sample of them
    (numpy seed 0, sorted indices), which depends only on the output's size."""
    import numpy as np
    import torch
    t = t.reshape(-1)
    if t.numel() > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
        t = t[torch.from_numpy(idx).to(t.device)]
    return t.to("cpu", torch.float64).numpy()


def write_outputs(path, outputs):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ CPU side (oracle)
def cpu_cg_rate(n_sample, iters, full_nnz, scale=True):
    """Times the oracle's CSR CG loop (the reference's loop, solver.py:144-229) on a Kuhn-cube Poisson operator of size
    n_sample built on the CPU, and scales the measured rate by nnz_sample/nnz_full to the benchmark workload (CG is
    memory-bound and linear in nnz far beyond the last-level cache).  Returns (iters/s at full size, description, cores)."""
    import numpy as np
    import torch
    from femb200 import meshgen
    from oracle import fem_oracle as O
    c, t = meshgen.kuhn_cube(n_sample)
    c, t = c.numpy(), t.numpy()
    Ke = O.c3d4_poisson_K(c, t)
    crow, col, val, n = O.assemble_csr(Ke, t, 1, c.shape[0])
    load = np.bincount(t.reshape(-1), weights=np.repeat(O.tet_volumes(c, t) / 4, 4), minlength=c.shape[0]).reshape(-1, 1)
    fixed = np.flatnonzero(c[:, 2] == 0)
    kind = "port"
    try:
        from oracle import c_oracle          # C + pthreads build of the same loop: all host cores
        threads = c_oracle.threads()
        impl = f"compiled oracle CG loop (C + pthreads, {threads} threads)"
        solve = lambda k: c_oracle.cg_csr(crow, col, val, load, fixed, tol=0.0, max_iter=k)  # noqa: E731
    except OSError:
        impl, threads = "numpy oracle CG loop", 1
        apply_fn = lambda v: O.csr_matvec(crow, col, val, v).reshape(-1, 1)  # noqa: E731
        solve = lambda k: O.cg_solve(apply_fn, load, fixed, tol=0.0, max_iter=k)  # noqa: E731
    solve(2)                                   # warm-up
    t0 = time.perf_counter()
    solve(iters)
    dt = time.perf_counter() - t0
    rate_sample = iters / dt
    desc = (f"{impl}; sample = {iters} CG iterations on the n={n_sample} Kuhn-cube Poisson operator ({t.shape[0]} tets, nnz {val.size}), "
            f"{rate_sample:.1f} it/s measured")
    if not scale:
        return rate_sample, desc + " (not extrapolated)", threads, kind
    rate_full = rate_sample * (val.size / full_nnz)
    desc += f", scaled by nnz ratio {val.size / full_nnz:.4f} to the full workload"
    return rate_full, desc, threads, kind


# ------------------------------------------------------------------------------------------------ BASELINE config 2 (secondary)
def config2(dev, hbm, n=69, iters=100):
    """P2 tet linear elasticity (BASELINE config 2: ~2 M C3D10 tets, fp64): element K, CSR assembly from Ke, block-CSR SpMV and
    Jacobi-PCG, each with its SURVEY 8d byte count against the measured HBM peak.  Reported beside the headline workload."""
    import torch
    import element as el
    from femb200 import meshgen, ops

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = ev(), ev()
        e0.record()
        out = None
        for _ in range(reps):
            out = None          # release the previous multi-GB result before the next call allocates
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, out

    c1, t1 = meshgen.kuhn_cube(n, device=dev)
    coords, e10 = meshgen.p1_to_p2_lattice(n, meshgen.swap01(t1), device=dev)
    del c1, t1
    M, N = e10.shape[0], coords.shape[0]
    ms_K, K = timed(lambda: el.compute_c3d10_K_matrix(coords, e10, 1.0, 0.3, device=dev, dtype=torch.float64))
    plan = el.CsrPlan(e10, N, dev)
    plan.pattern(3)
    vals = torch.empty(plan.nnz_nodes * 9, device=dev, dtype=torch.float64)
    ms_A, _ = timed(lambda: plan.assemble(K, 3, out=vals))
    del K
    nnz = vals.numel()
    brow, bcol = plan.pattern(1)
    A = ops.Bsr3.from_csr_values(brow, bcol, vals)
    x = torch.randn(3 * N, dtype=torch.float64, device=dev)
    ms_S, _ = timed(lambda: A.spmv(x), reps=10)
    mask = torch.ones((N, 3), dtype=torch.uint8, device=dev)
    mask[coords[:, 2] == 0] = 0
    mask = mask.reshape(-1).contiguous()
    F = torch.zeros((N, 3), dtype=torch.float64, device=dev)
    F[coords[:, 2] == 1, 2] = 1.0 / float((coords[:, 2] == 1).sum())
    minv = A.jacobi(mask)
    A.cg_solve(F, minv=minv, tol=0.0, max_iter=10, check_every=10)
    _, info = A.cg_solve(F, minv=minv, tol=0.0, max_iter=iters, check_every=min(iters, 50))
    ms_it = info["loop_ms"] / iters
    bytes_K = M * (10 * 8 + 900 * 8) + N * 24                  # SURVEY 8d: Ke materialised
    bytes_A = M * 900 * (8 + 4) + nnz * 8                       # SURVEY 8d: two-step assembly
    bytes_S_csr = nnz * 12 + 3 * N * 20                         # SURVEY 8d: scalar-CSR SpMV
    bytes_S_own = nnz * 8 + (nnz // 9) * 4 + N * 4 + 3 * N * 16  # what the 3x3 block layout moves
    frac = lambda b, ms: round(b / (ms * 1e-3) / 1e9 / hbm, 4)  # noqa: E731
    return {
        "workload": f"P2 tet linear elasticity, Kuhn n={n}: {M} C3D10 tets, {N} nodes, {3 * N} dofs, CSR nnz {nnz} (BASELINE config 2)",
        "element_K": {"ms": round(ms_K, 3), "elems_per_s": round(M / ms_K * 1e3), "algorithmic_bytes": bytes_K, "frac": frac(bytes_K, ms_K)},
        "assemble_from_Ke": {"ms": round(ms_A, 3), "elems_per_s": round(M / ms_A * 1e3), "algorithmic_bytes": bytes_A, "frac": frac(bytes_A, ms_A),
                             "kernel": "assemble_gather_batched<8,3,4>"},
        "assembled_elems_per_s": round(M / (ms_K + ms_A) * 1e3),
        "spmv_bsr3": {"ms": round(ms_S, 4), "bytes_moved": bytes_S_own, "frac_bytes_moved": frac(bytes_S_own, ms_S),
                      "algorithmic_bytes_scalar_csr": bytes_S_csr, "frac_scalar_csr_bytes": frac(bytes_S_csr, ms_S),
                      "kernel": "spmv_bsr3_vec_kernel (3x3 block-CSR, warp per block row)"},
        "jacobi_pcg": {"iters_per_s": round(1e3 / ms_it, 1), "ms_per_iter": round(ms_it, 4),
                       "algorithmic_bytes_scalar_csr": bytes_S_csr + 11 * 3 * N * 8, "frac_scalar_csr_bytes": frac(bytes_S_csr + 11 * 3 * N * 8, ms_it),
                       "frac_bytes_moved": frac(bytes_S_own + 11 * 3 * N * 8, ms_it)},
    }


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import element as el
    import solver as sv
    from femb200 import meshgen, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    torch.manual_seed(0)
    dev = torch.device(f"cuda:{local}")
    n = args.n
    K, W = args.steps, max(args.warmup, 3)
    outputs = {}            # --dump-outputs: name -> host array

    if world > 1:
        from femb200 import dist_cg
        if args.config == 2:
            return dist_cg.bench_config2(args, dev, rank, world, METRIC, UNIT)
        return dist_cg.bench(args, dev, rank, world, METRIC, UNIT)

    sampler = ClockSampler(local)          # started first: nvidia-smi needs up to a second before its first sample
    # ---- mesh + operator (resident in HBM before any timed region)
    coords, tets = meshgen.kuhn_cube(n, device=dev)
    M, N = tets.shape[0], coords.shape[0]
    t0 = time.perf_counter()
    plan = el.CsrPlan(tets, N, dev)
    torch.cuda.synchronize()
    t_plan = time.perf_counter() - t0
    crow, col = plan.pattern(1)
    vals = plan.assemble_c3d4(coords, "poisson")
    nnz = vals.numel()
    fixed = torch.nonzero(coords[:, 2] == 0).reshape(-1)
    mask = torch.ones(N, dtype=torch.uint8, device=dev)
    mask[fixed] = 0
    F = torch.full((N, 1), 1.0 / N, dtype=torch.float64, device=dev)
    hbm, peak_src = peaks()
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    # ---- assembly: fused coords -> CSR values, K passes
    for _ in range(W):
        plan.assemble_c3d4(coords, "poisson", out=vals, check_singular=False)
    a0, a1 = ev(), ev()
    reps_a = max(3, min(K, 10))
    torch.cuda.synchronize()
    a0.record()
    for _ in range(reps_a):
        plan.assemble_c3d4(coords, "poisson", out=vals, check_singular=False)
    a1.record()
    torch.cuda.synchronize()
    ms_asm = a0.elapsed_time(a1) / reps_a
    if args.dump_outputs:
        outputs["assembly_csr_values"] = dump_sample(vals)
    bytes_asm = M * 4 * 8 + N * 24 + nnz * 8          # SURVEY 8d: conn as the API receives it (int64) + coords + values
    # drop-in element matrices (compute_K_matrix path), Poisson 4x4
    Ke = el.compute_c3d4_poisson_K_matrix(coords, tets, device=dev, dtype=torch.float64)
    k0, k1 = ev(), ev()
    torch.cuda.synchronize()
    k0.record()
    for _ in range(3):      # the drop-in call as a user makes it in a loop: result written into the buffer it already owns
        el.compute_c3d4_poisson_K_matrix(coords, tets, device=dev, dtype=torch.float64, out=Ke)
    k1.record()
    torch.cuda.synchronize()
    ms_ke = k0.elapsed_time(k1) / 3
    Ke = None               # ... and as a fresh allocation per call (the previous result released first)
    torch.cuda.synchronize()
    k0.record()
    for _ in range(3):
        Ke = None
        Ke = el.compute_c3d4_poisson_K_matrix(coords, tets, device=dev, dtype=torch.float64)
    k1.record()
    torch.cuda.synchronize()
    ms_ke_alloc = k0.elapsed_time(k1) / 3
    bytes_ke = M * (4 * 8 + 16 * 8) + N * 24
    g0, g1 = ev(), ev()
    torch.cuda.synchronize()
    g0.record()
    for _ in range(3):
        plan.assemble(Ke, 1, out=vals)
    g1.record()
    torch.cuda.synchronize()
    ms_gather = g0.elapsed_time(g1) / 3
    del Ke
    plan.assemble_c3d4(coords, "poisson", out=vals, check_singular=False)

    # ---- dominant kernel alone: CSR SpMV, K launches on the current stream
    x = torch.randn(N, dtype=torch.float64, device=dev)
    for _ in range(W):
        ops.spmv(crow, col, vals, x)
    s0, s1 = ev(), ev()
    torch.cuda.synchronize()
    s0.record()
    for _ in range(K):
        ops.spmv(crow, col, vals, x)
    s1.record()
    torch.cuda.synchronize()
    ms_spmv = s0.elapsed_time(s1) / K
    bytes_spmv = nnz * 12 + N * 20                      # SURVEY 8d

    # ---- CG: W warm-up iterations, then exactly K timed iterations (tol=0 never converges)
    ops.cg_solve(crow, col, vals, F, mask=mask, tol=0.0, max_iter=max(W, 50), check_every=50)
    torch.cuda.synchronize()
    c0, c1 = ev(), ev()
    c0.record()
    u, info = ops.cg_solve(crow, col, vals, F, mask=mask, tol=0.0, max_iter=K, check_every=min(K, 50))
    c1.record()
    torch.cuda.synchronize()
    ms_call = c0.elapsed_time(c1)
    ms_loop = info["loop_ms"]
    assert info["iterations"] == K, info
    if args.dump_outputs:
        outputs["cg_u"] = dump_sample(u)
        outputs["cg_rs"] = np.array([info["rs"]], dtype=np.float64)
    bytes_iter = bytes_spmv + 9 * N * 8                 # SURVEY 8d

    # ---- e2e: public solver API, load vector from pinned host memory, solution read back to the host
    F_host = torch.full((N, 1), 1.0 / N, dtype=torch.float64).pin_memory()
    u_host = torch.empty((N, 1), dtype=torch.float64).pin_memory()
    A = torch.sparse_csr_tensor(crow, col, vals, size=(N, N))

    def e2e_call():
        e0, e1 = ev(), ev()
        torch.cuda.synchronize()
        e0.record()
        u2 = sv.stable_conjugate_gradient_solver(A, tets, F_host.to(dev, non_blocking=True), fixed, tol=0.0, max_iter=K, device=dev, verbose=False)
        u_host.copy_(u2, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), u2

    # the first call of this path is timed too and reported (`first_call_ms`: it pays the solver's one-time setup for this
    # operator); the e2e value is the median of repeated calls, EVERY one of which copies F in and u out, until >= 50 ms are timed
    ms_e2e_first, u2 = e2e_call()
    e2e_ms = []
    while (sum(e2e_ms) < 50.0 or len(e2e_ms) < 3) and len(e2e_ms) < 25:
        ms_c, u2 = e2e_call()
        e2e_ms.append(ms_c)
    e2e_ms.sort()
    ms_e2e = e2e_ms[len(e2e_ms) // 2]
    if args.dump_outputs:
        outputs["e2e_u"] = dump_sample(u_host)
    t_soak = time.perf_counter()           # untimed: keep the same loop running until the sampler has >= 0.5 s under load
    while time.perf_counter() - t_soak < 0.5:
        ops.cg_solve(crow, col, vals, F, mask=mask, tol=0.0, max_iter=200, check_every=50)
    clocks = sampler.stop()
    # ---- topology on the same mesh (bit-exact face lists; buckets by smallest node + in-warp sort, csrc/topology.cu)
    topo = None
    if not args.no_topo:
        try:
            ops.entities(ops.ENT_TET_FACES, tets, dev)             # warm-up (scratch pool, cub temp sizes)
            t0e, t1e = ev(), ev()
            torch.cuda.synchronize()
            t0e.record()
            faces, extra, pairs = ops.entities(ops.ENT_TET_FACES, tets, dev)
            t1e.record()
            torch.cuda.synchronize()
            ms_topo = t0e.elapsed_time(t1e)
            bytes_topo = M * 4 * 8 + faces.numel() * 8 + extra.numel() * 8 + pairs.numel() * 8   # SURVEY 8d: conn in, face lists out
            topo = {"what": "tet surface faces + fourth node and shared-face pairs in one pass (faces bucketed by smallest node, one warp sorts a bucket)",
                    "ms": round(ms_topo, 2), "elems_per_s": round(M / (ms_topo * 1e-3), 1), "surface_faces": int(faces.shape[0]),
                    "shared_pairs": int(pairs.shape[0]), "algorithmic_bytes": bytes_topo,
                    "frac": round(bytes_topo / (ms_topo * 1e-3) / 1e9 / hbm, 4),
                    "note": "bucket records (12 B per face written, read once) and per-bucket pair lists are implementation overhead, not counted"}
            del faces, extra, pairs
        except Exception as exc:  # noqa: BLE001
            topo = {"error": f"{type(exc).__name__}: {exc}"}
    c2 = None
    if not args.no_c2:
        del A, u, u2, x, vals, crow, col, plan, coords, tets
        torch.cuda.empty_cache()
        try:
            c2 = config2(dev, hbm)
        except Exception as exc:  # noqa: BLE001  (the headline line must print regardless)
            c2 = {"error": f"{type(exc).__name__}: {exc}"}

    value = K / (ms_loop * 1e-3)
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": round(ms_loop / K, 5), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(n, M, N, nnz),
        "impl_details": {"index_dtype": "int32 CSR / int64 API connectivity", "partition": "none (1 GPU)"},
        "clocks": clocks,
        "e2e": {"value": round(K / (ms_e2e * 1e-3), 2), "unit": UNIT, "h2d_bytes_per_step": int(F_host.numel() * 8 / K),
                "d2h_bytes_per_step": int(u_host.numel() * 8 / K),
                "calls": len(e2e_ms), "first_call_ms": round(ms_e2e_first, 3), "ms_per_call": round(ms_e2e, 3),
                "note": f"one solver-API call of {K} iterations: F pinned host -> device, CG, u -> pinned host; bytes are per call / K; "
                        "median over `calls` identical calls after one untimed-in-the-median first call"},
        "gpu_launches": (3 if os.environ.get("FEMB_CG_CLASSIC") else 2) * K + 4,
        "roofline": {"kernel": "spmv_tma_kernel<1,false> (TMA-pipelined CSR SpMV; its fused twin is CG step k1)", "bound": "hbm",
                     "achieved": round(bytes_spmv / (ms_spmv * 1e-3) / 1e9, 1), "peak": hbm, "unit": "GB/s",
                     "frac": round(bytes_spmv / (ms_spmv * 1e-3) / 1e9 / hbm, 4), "traffic": ncu_traffic(n, "spmv_tma_kernel"), "peak_source": peak_src,
                     "traffic_source": "profiles/r02_traffic.json (ncu --set full capture of this kernel on this workload; null for other sizes)",
                     "ms_per_launch": round(ms_spmv, 4), "algorithmic_bytes": bytes_spmv},
        "cg_iteration": {"ms": round(ms_loop / K, 4), "algorithmic_bytes": bytes_iter,
                         "achieved_GBps": round(bytes_iter / (ms_loop / K * 1e-3) / 1e9, 1),
                         "frac": round(bytes_iter / (ms_loop / K * 1e-3) / 1e9 / hbm, 4), "api_call_ms": round(ms_call, 2),
                         "kernels": "spmv_tma_kernel<1,true> (SpMV + p.Ap, r.Ap, Ap.Ap -> alpha, rs_new, beta) + cg_merged_kernel "
                                    "(u, r, p in one pass + exact r.r): 2 launches, 7 vector passes + r in the SpMV",
                         "bytes_actually_moved": bytes_spmv + 8 * N * 8},
        "assembly": {"metric": "assembled_elems_per_s", "value": round(M / (ms_asm * 1e-3), 1), "ms": round(ms_asm, 3),
                     "kernel": "pad_coords + assemble_p1_poisson_tiles (coords -> CSR values; pattern and per-incidence records prebuilt)",
                     "algorithmic_bytes": bytes_asm, "achieved_GBps": round(bytes_asm / (ms_asm * 1e-3) / 1e9, 1),
                     "frac": round(bytes_asm / (ms_asm * 1e-3) / 1e9 / hbm, 4),
                     # SURVEY 8d lists the slot map (M*nd^2*4 bytes) as an add-on when one is read; this kernel reads a
                     # 16-byte record per incidence (the three other node ids + their slots) instead of conn + slot map
                     "algorithmic_bytes_with_slot_map": bytes_asm + M * 16 * 4,
                     "frac_with_slot_map": round((bytes_asm + M * 16 * 4) / (ms_asm * 1e-3) / 1e9 / hbm, 4),
                     "traffic": ncu_traffic(n, "assemble_p1_poisson_tiles"), "plan_build_s": round(t_plan, 3),
                     "element_K_elems_per_s": round(M / (ms_ke * 1e-3), 1), "element_K_GBps": round(bytes_ke / (ms_ke * 1e-3) / 1e9, 1),
                     "element_K_frac": round(bytes_ke / (ms_ke * 1e-3) / 1e9 / hbm, 4), "element_K_ms": round(ms_ke, 3),
                     "element_K_ms_with_fresh_allocation": round(ms_ke_alloc, 3),
                     "two_step_gather_ms": round(ms_gather, 3)},
    }
    if topo is not None:
        out["topology"] = topo
    if c2 is not None:
        out["config2"] = c2
    if not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline_leg(args, nnz)
    print(json.dumps(out), flush=True)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)


def cpu_baseline_leg(args, nnz):
    """cpu_baseline of the GPU arm (rank 0, N=1): the reference itself on a bounded sample (kind "reference", measured, not
    extrapolated), with the compiled C port of the same loop on the same sample beside it as a second, labelled line."""
    n_s, iters = args.cpu_base_n, args.cpu_base_iters
    ref = None
    try:
        ref = reference_sample(n_s, iters)
    except Exception as exc:  # noqa: BLE001
        ref_err = f"{type(exc).__name__}: {exc}"
    port_rate, port_desc, port_cores, _ = cpu_cg_rate(n_s, max(iters, 20), nnz, scale=False)
    port = {"value": round(port_rate, 3), "unit": UNIT, "cores": port_cores, "kind": "port", "sample": port_desc}
    if ref is None:
        port["note"] = "reference not installed on this box (baseline/_ref missing): this is the C port, not the reference" if "ref_err" not in locals() else ref_err
        return port
    return {"value": round(ref["rate"], 3), "unit": UNIT, "cores": ref["threads"], "kind": "reference",
            "sample": (f"UNMODIFIED reference (baseline/_ref/solver: stable_conjugate_gradient_solver, torch CPU {ref['threads']} threads, fp64): "
                       f"{iters} CG iterations on the n={n_s} Kuhn-cube Poisson sample ({ref['tets']} tets), measured, not extrapolated; "
                       "the full-size reference arm is `bench.py --impl reference`"),
            "ms_per_iter": round(ref["ms_per_iter"], 2), "port": port}


def workload_config(n, M, N, nnz):
    """The `config` object, identical on both arms (the driver compares them)."""
    return {"workload": f"P1 tet Poisson, Kuhn cube n={n}: {M} C3D4 tets, {N} nodes, CSR nnz {nnz} (BASELINE config 4); "
                        "step = one CG iteration of the reference loop (solver.py:144-229)",
            "tol": 0.0,
            "l2": "inputs larger than the last-level cache on both arms (GPU arm: CSR operator %.2f GB vs 126 MB L2, never flushed "
                  "artificially; reference arm: per-element matrices of the sample, GBs vs tens of MB of L3)" % (nnz * 12 / 1e9)}


def kuhn_counts(n):
    N = (n + 1) ** 3
    M = 6 * n ** 3
    edges = 3 * n * (n + 1) ** 2 + 3 * n * n * (n + 1) + n ** 3  # axis + face-diagonal + body-diagonal edges of the Kuhn cube
    return M, N, N + 2 * edges


def reference_sample(n_sample, iters, c1=False, timeout=1500):
    """Times the UNMODIFIED reference (baseline/_ref/solver, torch CPU, all host threads) in a subprocess: its
    `stable_conjugate_gradient_solver` on the n_sample Kuhn-cube Poisson problem (baseline/ref_arm.py).  None if the
    reference is not installed on this box."""
    arm = os.path.join(ROOT, "baseline", "ref_arm.py")
    if not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "solver", "solver.py")):
        return None
    cmd = [sys.executable, arm, "--n", str(n_sample), "--iters", str(iters)] + (["--c1"] if c1 else [])
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):   # torchrun pins OMP_NUM_THREADS=1
        env.pop(k, None)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    if r.returncode != 0:
        raise RuntimeError(f"reference arm failed: {r.stderr[-400:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def run_reference(args):
    """`--impl reference`: the reference's own torch-CPU CG (solver.py:144-229 driving element.py:429-464) on the box's host
    cores.  `value` is the MEASURED rate on the bounded sample (n = --cpu-n), never extrapolated; a second, smaller sample and
    BASELINE config 1 (run exactly) are printed beside it so the size dependence is visible."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.n
    M, N, nnz = kuhn_counts(n)
    K, W = args.steps, max(args.warmup, 3)
    iters = max(3, min(K, args.cpu_iters))
    t0 = time.perf_counter()
    big = reference_sample(args.cpu_n, iters, c1=True)
    if big is None:      # reference not installed on this box: fall back to the labelled C port (never silently)
        rate, desc, cores, kind = cpu_cg_rate(args.cpu_n, iters, nnz, scale=False)
        extra = {"note": "baseline/_ref missing on this box: value is the C port of the reference loop on the sample, NOT the reference"}
    else:
        small_n = max(20, args.cpu_n // 2)
        small = reference_sample(small_n, iters)
        rate, cores, kind = big["rate"], big["threads"], "reference"
        Ms = big["tets"]
        desc = (f"UNMODIFIED reference (baseline/_ref/solver: stable_conjugate_gradient_solver -> compute_nodal_forces, torch {cores} threads, "
                f"fp64): {iters} CG iterations (after 1 warm-up) on the n={args.cpu_n} Kuhn-cube Poisson sample = {Ms} tets "
                f"({Ms / M:.4f} of the workload's {M}), measured {rate:.3f} it/s; value is NOT extrapolated to the full mesh")
        per_tet = [big["ms_per_iter"] * 1e6 / big["tets"], small["ms_per_iter"] * 1e6 / small["tets"]]
        extra = {"reference_measurements": {
            "sample": {k: big[k] for k in ("n", "tets", "nodes", "iters", "rate", "ms_per_iter", "setup_s", "threads")},
            "half_sample": {k: small[k] for k in ("n", "tets", "nodes", "iters", "rate", "ms_per_iter", "setup_s", "threads")},
            "ns_per_tet_iteration": [round(v, 2) for v in per_tet],
            "config1_exact": big.get("c1"),
            "full_size_estimate": {"iters_per_s": round(1e3 / (per_tet[0] * 1e-6 * M), 4),
                                   "how": "linear in tets from the larger sample (ns per tet-iteration above); an ESTIMATE, not `value`"}}}
    out = {"impl": "reference", "metric": METRIC, "value": round(rate, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
           "ms_per_step": round(1e3 / rate, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
           "data": "synthetic", "config": workload_config(n, M, N, nnz),
           "cpu_baseline": {"value": round(rate, 3), "unit": UNIT, "cores": cores, "kind": kind, "sample": desc},
           "e2e": {"value": round(rate, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "host": {"cpu_count": os.cpu_count(), "cpu_model": cpu_model()},
           "wall_s": round(time.perf_counter() - t0, 1)}
    out.update(extra)
    print(json.dumps(out), flush=True)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--n", type=int, default=220, help="Kuhn cube cells per edge (220 -> 63.9M tets)")
    ap.add_argument("--impl", default="femb200", choices=["femb200", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[4, 2], help="BASELINE config: 4 = P1 Poisson 64 M tets (headline); "
                    "2 = P2 elasticity 2 M tets, Jacobi-PCG (multi-GPU line: torchrun ... bench.py --gpus N --config 2)")
    ap.add_argument("--n2", type=int, default=69, help="Kuhn cube cells per edge of config 2 (69 -> 1.97 M C3D10 tets)")
    ap.add_argument("--cpu-n", type=int, default=96, help="cube size of the CPU sample")
    ap.add_argument("--cpu-iters", type=int, default=20)
    ap.add_argument("--cpu-base-n", type=int, default=64, help="cube size of the cpu_baseline sample inside the GPU arm (~10 s of CPU work)")
    ap.add_argument("--cpu-base-iters", type=int, default=10)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-topo", action="store_true", help="skip the face-connectivity timing on the headline mesh")
    ap.add_argument("--no-c2", action="store_true", help="skip the secondary BASELINE config 2 (P2 elasticity) measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed paths' last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "femb200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is supported on the single-GPU femb200 arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
