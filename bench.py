#!/usr/bin/env python
"""bench.py -- ExactGP MLL evaluations/s (and fused K.V GF/s) at the BASELINE C2 workload.

A "step" = one evaluation of the exact-GP marginal log likelihood through the BBMM path: pivoted-Cholesky
preconditioner (rank 100) -> N(0,P) probes -> mBCG (t = 10 probes + y, J = 21 iterations) -> SLQ log-det ->
log_prob, on synthetic data (BASELINE.md section 2): X ~ U[0,1]^{N x d}, y = sin(3 sum x) + 0.1 eps, RBF.

    python bench.py --gpus 1 --steps 10 --warmup 3            # our engine (libgpbbmm, sm_100a)
    python bench.py --impl reference --steps 2 --warmup 1     # the reference algorithm on the host CPU cores, full N
    torchrun ... bench.py --gpus N ...                        # rows of K sharded over N GPUs (strong scaling)
    python bench.py --steps 10 --warmup 3 --dump-outputs DIR  # + what the last timed step returned, as DIR/<name>.npy

Rank 0 prints ONE JSON line (see the task contract): value = whole-job MLL evals/s with inputs resident in HBM,
e2e = same metric through the public gpytorch-style API with HOST inputs (H2D of X, y and D2H of the result
inside the timed region), roofline = the fused K.V kernel alone (CUDA events on its own stream), cpu_baseline =
the oracle port on the host cores, ONE evaluation at the full configuration (never a scaled sample),
parity_at_config = our result against that evaluation (same inputs, same probe base samples), c3 = the same
measurement at BASELINE configs[2] (N = 200 000, Matern-5/2, d = 20) on the same ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line.  Libraries print to fd 1 behind Python's back (NCCL's version banner under
# NCCL_DEBUG=VERSION/INFO, torchrun notices), so fd 1 is pointed at stderr for the whole run and the JSON line is written to the
# saved original stdout; NCCL_DEBUG is left as the caller set it.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


WORKLOADS = {
    # BASELINE.json configs[0]: the reference's own CPU-runnable case (N < min_preconditioning_size: no preconditioner,
    # Rademacher probes; N > max_cholesky_size = 800: the mBCG path)
    "c1": dict(name="ExactGP RBF N=1000 d=3, mBCG t=11 probes, no preconditioner (N < 2000)", n=1000, d=3, kind="rbf",
               lengthscale=0.5, outputscale=1.0, noise=0.1, probes=10, rank=15),
    # BASELINE.json configs[1]: the configuration the metric is quoted on
    "c2": dict(name="ExactGP RBF N=50000 d=10, mBCG t=11 probes + rank-100 pivoted-Cholesky precond", n=50000, d=10,
               kind="rbf", lengthscale=1.0, outputscale=1.0, noise=0.1, probes=10, rank=100),
    # configs[2]: the 8-GPU strong-scaling case
    "c3": dict(name="ExactGP Matern-5/2 N=200000 d=20, row-sharded K.V + NCCL CG dots", n=200000, d=20,
               kind="matern52", lengthscale=2.0, outputscale=1.0, noise=0.1, probes=10, rank=100),
    # configs[3]: batch of 16 independent exact GPs (own hyper-parameters per element), evaluated concurrently
    "c4": dict(name="Batched ExactGP (batch=16) RBF N=10000 d=8 -- batched Krylov / inv_quad_logdet path", n=10000, d=8, kind="rbf",
               lengthscale=0.9, outputscale=1.0, noise=0.1, probes=10, rank=100, batch=16),
    # configs[4]: SKI / KISS-GP, cubic interpolation onto a 100^3 grid (no preconditioner: Rademacher probes)
    "c5": dict(name="SKI/KISS-GP RBF N=1e6 d=3, grid 100^3 -- InterpolatedLinearOperator / Toeplitz matmul path", n=1000000, d=3, kind="rbf",
               lengthscale=0.2, outputscale=1.0, noise=0.1, probes=10, rank=0, grid=[100, 100, 100]),
    # small case for quick checks (not a BASELINE config)
    "small": dict(name="ExactGP RBF N=4000 d=3 (quick check, not a BASELINE config)", n=4000, d=3, kind="rbf", lengthscale=0.5,
                  outputscale=1.0, noise=0.1, probes=10, rank=15),
}
METRIC = "exactgp_mll_evals_per_sec"
UNIT = "evals/s"


def host_cores() -> int:
    """Usable host cores: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() over-reports inside a
    container and 128 torch threads on a few real cores run ~80x slower than 8)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    env = os.environ.get("GP_CPU_THREADS")
    return int(env) if env else n


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# synthetic inputs (BASELINE.md section 2).  Kept here (not imported from oracle/) so that the product arm imports
# nothing from the oracle; tests/test_host_logic.py checks these against oracle.mll bit for bit.
# ------------------------------------------------------------------------------------------------------------
def synthetic_problem(n, d, seed=0):
    """X ~ U[0,1]^{n x d}, y = sin(3 sum_d x) + 0.1 eps (fp64 draw, cast to fp32)."""
    import torch

    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    y = torch.sin(3 * x.sum(-1)) + 0.1 * torch.randn(n, generator=g, dtype=torch.float64)
    return x.float(), y.float()


def make_probe_noise(n, k, tp, seed):
    """Base samples shared by the CPU and GPU arms: eps1 [k,tp], eps2 [n,tp] ~ N(0,1) (z = L eps1 + sigma eps2),
    rademacher [n,tp]."""
    import torch

    g = torch.Generator().manual_seed(seed)
    eps1 = torch.randn(max(k, 1), tp, generator=g, dtype=torch.float64).float()
    eps2 = torch.randn(n, tp, generator=g, dtype=torch.float64).float()
    rad = torch.randint(0, 2, (n, tp), generator=g).float() * 2 - 1
    return eps1, eps2, rad


# ------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port (torch on the host cores) at the FULL configuration, never scaled
# ------------------------------------------------------------------------------------------------------------
def cpu_reference_eval(w, n_rows=None, seed=0):
    """One full MLL evaluation of the reference algorithm (dense K once + mBCG with dense K @ V) on the first n_rows
    rows of the workload (default: all of them).  Returns (seconds, oracle result)."""
    import torch
    import warnings
    from oracle import mll as om

    n = w["n"] if n_rows is None else n_rows
    x, y = synthetic_problem(n, w["d"], seed)
    pn = make_probe_noise(n, w["rank"], w["probes"], 1)
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r = om.mll_bbmm(w["kind"], x, y, 0.0, w["lengthscale"], w["outputscale"], w["noise"], pn, precond_size=w["rank"])
    return time.perf_counter() - t0, r


def tune_threads(w):
    """Pick the torch thread count that runs the reference path fastest on this host (<= usable cores)."""
    import torch

    cores = host_cores()
    cands = sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores}, reverse=True)
    best, best_t = cores, None
    for c in cands:
        torch.set_num_threads(c)
        cpu_reference_eval(w, min(w["n"], 1500))
        t, _ = cpu_reference_eval(w, min(w["n"], 3000))
        if best_t is None or t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def dense_fits(w):
    """The reference materialises K (lazy_evaluated_kernel_tensor.py:343-373): N^2 fp32 plus one N^2 temporary."""
    need = 2.2 * 4.0 * w["n"] ** 2 * (1.0 if w["kind"] == "rbf" else 2.5)
    try:
        import psutil
        return need < 0.8 * psutil.virtual_memory().available
    except Exception:
        return need < 48e9


def cpu_baseline(w):
    """ONE evaluation of the oracle port at the full configuration on the host cores (C2: ~10 s, 20 GB of host RAM)."""
    cores = tune_threads(w)
    if not dense_fits(w):
        return {"value": None, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"skipped: dense K at N={w['n']} does not fit in host memory (the reference would need its chunked path)"}
    dt, r = cpu_reference_eval(w)
    return {
        "value": 1.0 / dt, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"oracle port (torch CPU fp32, {cores} threads): dense K once + mBCG with dense K@V, ONE evaluation at the "
                  f"full configuration N={w['n']} ({dt:.2f} s); no scaling",
        "sample_seconds": dt, "sample_rows": w["n"], "cg_iters": r.iters,
        "mll": r.mll, "inv_quad": r.inv_quad, "logdet": r.logdet,
    }


def run_reference(args, w):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = tune_threads(w)
    if not dense_fits(w):
        emit({"impl": "reference", "unavailable": f"dense K at N={w['n']} does not fit in this host's memory; "
              "the reference's default path materialises K (lazy_evaluated_kernel_tensor.py:343-373)"})
        return
    # every step is ONE evaluation at the full configuration (never a scaled sample).  All requested steps run; the requested
    # warm-up count is honoured as long as the run stays within ~5 minutes, beyond that it is cut and the line says so.
    t_probe, r = cpu_reference_eval(w)            # also the first warm-up evaluation
    budget = float(os.environ.get("GP_REF_BUDGET_S", 300.0))
    warm = max(0, min(args.warmup - 1, int((budget - args.steps * t_probe) / t_probe) - 1))
    steps = args.steps
    for _ in range(warm):
        cpu_reference_eval(w)
    times = []
    for _ in range(steps):
        dt, r = cpu_reference_eval(w)
        times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    val = 1e3 / ms
    sample = (f"oracle port of the reference path (gpytorch kernels + linear_operator mBCG restated, torch CPU fp32, {cores} threads): "
              f"every step is one full evaluation at N={w['n']} (dense K once + {r.iters} dense K@V); no scaling")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": 1 + warm, "steps_requested": args.steps, "warmup_requested": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["name"], "parallelism": "host cpu", "timing": "perf_counter around each full evaluation",
                   "lengthscale": w["lengthscale"], "outputscale": w["outputscale"], "noise": w["noise"],
                   "cg_iters": r.iters, "mll": r.mll, "inv_quad": r.inv_quad, "logdet": r.logdet},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mll": r.mll, "log_prob": r.log_prob, "inv_quad": r.inv_quad, "logdet": r.logdet,
                                         "cg_iters": r.iters})


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
def dump_outputs(path, arrays):
    """--dump-outputs: one path/<name>.npy per returned value, float32 arrays as they are and everything else as float64, so
    that runs of two builds on the same (seeded) inputs can be compared value for value."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(path, f"{name}.npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def mll_result_arrays(res, t, prefix=""):
    """The fields of the MllResult Plan.mll returns; resid holds one CG residual norm per right-hand side (t of them)."""
    out = {k: getattr(res, k) for k in ("mll", "log_prob", "inv_quad", "logdet", "logdet_precond", "cg_iters", "tridiag_size",
                                        "precond_rank", "status_flags")}
    out["resid"] = [float(v) for v in res.resid[:t]]
    return {prefix + k: v for k, v in out.items()}


MLL_KNOBS = dict(min_precond_size=2000, precond_tol=1e-3, cg_tol=1.0, max_cg_iter=1000, max_tridiag_iter=20)  # reference defaults


def measure_workload(w, args, env, steps, warmup, sample_clocks=False):
    """Device-resident timing of `steps` MLL evaluations of workload `w` (+ the fused K.V kernel alone).
    env = (rank, world, local, dev, comm, dist).  Returns a dict; every rank takes part, rank 0's copy is printed."""
    import torch

    from gpytorch_b200.distributed import shard_rows
    from gpytorch_b200.engine import Plan

    rank, world, local, dev, comm, dist = env
    n, d = w["n"], w["d"]
    rb, rc, _ = shard_rows(n, world, rank)
    x, y = synthetic_problem(n, d, 0)
    eps1, eps2, rad = make_probe_noise(n, w["rank"], w["probes"], 1)
    xd = x.to(dev)
    e1d, e2d, radd = eps1.to(dev), eps2[rb : rb + rc].contiguous().to(dev), rad[rb : rb + rc].contiguous().to(dev)
    y_loc = y[rb : rb + rc].contiguous().to(dev)
    plan = Plan(xd, backend=args.backend, row_begin=rb, row_count=rc if world > 1 else 0, comm=comm)
    if "grid" in w:
        # GridInterpolationKernel(grid_size, grid_bounds=[(0, 1)]^d): utils/grid.py:142-180 extends the bounds by one cell
        axes = [torch.linspace(0.0 - 1.0 / (g - 2), 1.0 + 1.0 / (g - 2), g) for g in w["grid"]]
        plan.set_ski(w["grid"], [float(a[0]) for a in axes], [float(a[1] - a[0]) for a in axes])
    plan.set_hypers(w["kind"], w["lengthscale"], w["outputscale"], w["noise"])
    info = plan.info()
    l2_flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step():
        l2_flush.zero_()  # evict the L2 between steps (timing rule); ~60 us of the step
        res, _ = plan.mll(y_loc, e1d, e2d, radd, w["probes"], w["rank"], MLL_KNOBS["min_precond_size"], MLL_KNOBS["precond_tol"],
                          MLL_KNOBS["cg_tol"], MLL_KNOBS["max_cg_iter"], MLL_KNOBS["max_tridiag_iter"], warn=False)
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        res = step()
    barrier()
    sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    l0 = plan.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        res = step()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = plan.launches() - l0
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / steps

    # ---- the fused K.V kernel alone: roofline ----
    v = torch.randn(n, w["probes"] + 1, device=dev)
    kms = plan.time_kmv_kernel(v, warmup=3, reps=20)
    tt = w["probes"] + 1
    flops = 2.0 * rc * n * (d + tt)  # algorithmic flops of this rank's row block (SURVEY.md section 8d)
    peaks, peak_src = measured_peaks()
    ach = flops / (kms * 1e-3) / 1e12
    peak = float(peaks["bf16_tflops"])
    trans = (2 if w["kind"] != "rbf" else 1) * rc * n  # transcendental ops per launch (ex2, + sqrt for Matern)
    mufu_peak = 16.0 * info["n_sm"] * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6  # 16 MUFU/clk/SM (tools/mufu_bench.cu: 15.99)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "kmv_tc2_dram_bytes.json")
    if os.path.exists(tpath) and world == 1 and w is WORKLOADS["c2"] and info["backend"] == "tcgen05":
        with open(tpath) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    if info["backend"] == "ski":
        nnz = 4 ** d
        abytes = float(n) * nnz * (4 + 8)          # SURVEY.md section 8f: W stored as (int64 index, fp32 value) per non-zero
        hbm = float(peaks["hbm_gbs"])
        roofline = {"bound": "hbm", "kernel": "gp::ski_scatter / ski_mode / ski_gather (one K_ski.V product)", "achieved": abytes / (kms * 1e-3) / 1e9,
                    "peak": hbm, "unit": "GB/s", "frac": abytes / (kms * 1e-3) / 1e9 / hbm, "traffic": None, "peak_source": f"stream copy, {peak_src}",
                    "ms_per_launch": kms, "algorithmic_bytes_per_launch": abytes,
                    "note": "algorithmic bytes = N 4^d (4 + 8) B, the explicit W of the reference; the engine keeps W in compact per-dimension "
                            "form (20 d B per row), so achieved > peak is possible"}
        return {"value": 1e3 / ms_step, "ms_per_step": ms_step, "launches": int(launches), "clocks": clocks, "roofline": roofline,
                "info": info, "res": res, "flops": 0.0, "kms": kms,
                "ctx": dict(plan=plan, x=x, y=y, xd=xd, y_loc=y_loc, e1d=e1d, e2d=e2d, radd=radd, rb=rb, rc=rc, l2_flush=l2_flush, barrier=barrier)}
    roofline = {
        "bound": "tensor", "kernel": info.get("kernel", "gp::v2::kmv_tc2_kernel" if info["backend"] == "tcgen05" else "gp::kmv_simt_kernel"),
        "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
        "peak_source": f"bf16 dense burst, {peak_src}; the kernel runs kind::tf32 (nominal half of bf16) with a 3xTF32 split",
        "ms_per_launch": kms, "algorithmic_flops_per_launch": flops,
        "gpairs_per_s": rc * n / (kms * 1e-3) / 1e9,
        "mufu_bound": {"transcendentals_per_launch": trans, "achieved_per_s": trans / (kms * 1e-3),
                       "peak_per_s_at_max_clock": mufu_peak, "frac": trans / (kms * 1e-3) / mufu_peak,
                       "note": "all-MUFU ceiling; the kernel evaluates part of the ex2 on the FMA pipe, so frac may exceed 1"},
        "algorithmic_bytes_per_launch": 4.0 * (n * d + 2 * n * tt),
    }
    out = {
        "value": 1e3 / ms_step, "ms_per_step": ms_step, "launches": int(launches), "clocks": clocks, "roofline": roofline,
        "info": info, "res": res, "flops": flops, "kms": kms,
        "ctx": dict(plan=plan, x=x, y=y, xd=xd, y_loc=y_loc, e1d=e1d, e2d=e2d, radd=radd, rb=rb, rc=rc, l2_flush=l2_flush, barrier=barrier),
    }
    return out


def result_config(w, world, m):
    res, info = m["res"], m["info"]
    return {
        "workload": w["name"], "parallelism": f"row-shard x{world}" if world > 1 else "single GPU",
        "kind": w["kind"], "lengthscale": w["lengthscale"], "outputscale": w["outputscale"], "noise": w["noise"],
        "num_probes": w["probes"], "precond_rank_requested": w["rank"], **{k: v for k, v in MLL_KNOBS.items()},
        "backend": info["backend"], "nsplit": info["nsplit"], "kpad": info["kpad"],
        "l2_policy": "L2 flushed between timed steps by a 192 MiB memset inside the timed region",
        "cg_iters": res.cg_iters, "precond_rank": res.precond_rank, "tridiag_size": res.tridiag_size,
        "mll": res.mll, "inv_quad": res.inv_quad, "logdet": res.logdet,
        "kv_gflops_algorithmic": m["flops"] / (m["kms"] * 1e-3) / 1e9 * world,
    }


def run_c4(args, w):
    """BASELINE configs[3]: batch of `batch` independent exact GPs through the public API (batch_shape kernels / likelihood /
    MultivariateNormal.log_prob -> [B]); the elements run concurrently, one engine plan + CUDA stream each.  One step = one
    batched MLL evaluation (all B problems); value counts evaluations of single problems per second."""
    import torch

    import gpytorch_b200 as gp
    from gpytorch_b200 import settings

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, n, d = w["batch"], w["n"], w["d"]
    g = torch.Generator().manual_seed(0)
    X = torch.rand(B, n, d, generator=g)
    Y = torch.sin(3 * X.sum(-1)) + 0.1 * torch.randn(B, n, generator=g)
    bs = torch.Size([B])
    lik = gp.likelihoods.GaussianLikelihood(batch_shape=bs).to(dev)
    lik.noise = (w["noise"] * (1 + 0.05 * torch.arange(B))).unsqueeze(-1)

    class Model(gp.models.ExactGP):
        def __init__(self, tx, ty):
            super().__init__(tx, ty, lik)
            self.mean_module = gp.means.ZeroMean(batch_shape=bs)
            self.covar_module = gp.kernels.ScaleKernel(gp.kernels.RBFKernel(batch_shape=bs), batch_shape=bs)

        def forward(self, xx):
            return gp.distributions.MultivariateNormal(self.mean_module(xx), self.covar_module(xx))

    Xd, Yd = X.to(dev), Y.to(dev)
    model = Model(Xd, Yd).to(dev)
    model.covar_module.base_kernel.lengthscale = (w["lengthscale"] * (1 + 0.02 * torch.arange(B))).reshape(B, 1, 1)
    model.covar_module.outputscale = w["outputscale"] * (1 + 0.03 * torch.arange(B))
    mll = gp.mlls.ExactMarginalLogLikelihood(lik, model)
    model.train(); lik.train()
    l2_flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step():
        l2_flush.zero_()
        with torch.no_grad(), settings.max_preconditioner_size(w["rank"]), settings.num_trace_samples(w["probes"]), \
                settings.backend(args.backend), settings.probe_seed(1):
            return mll(model(Xd), Yd)

    for _ in range(args.warmup):
        out = step()
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms_step = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop()
    line = {
        "metric": METRIC, "value": B * 1e3 / ms_step, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["name"], "batch": B, "parallelism": "single GPU, one plan + stream per batch element, 16 host threads",
                   "kind": w["kind"], "precond_rank_requested": w["rank"], "num_probes": w["probes"],
                   "l2_policy": "L2 flushed between timed steps by a 192 MiB memset inside the timed region",
                   "step": "one batched MLL evaluation = 16 problems; value = single-problem evaluations per second",
                   "mll_per_element": [float(v) for v in out.tolist()]},
        "clocks": clocks, "e2e": None, "gpu_launches": None, "roofline": None, "cpu_baseline": None,
    }
    emit(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mll": out.detach().cpu().numpy()})


def run_ours(args, w):
    import torch
    import torch.distributed as dist

    import gpytorch_b200 as gp
    from gpytorch_b200 import settings
    from gpytorch_b200.distributed import Comm, init_from_env
    from gpytorch_b200.engine import Plan

    rank, world, local = init_from_env()
    dev = torch.device("cuda", local)
    if w["n"] % world:
        raise SystemExit(f"N={w['n']} must be divisible by the number of GPUs ({world})")
    comm = Comm(rank, world) if world > 1 else None
    env = (rank, world, local, dev, comm, dist)

    m = measure_workload(w, args, env, args.steps, args.warmup, sample_clocks=True)
    c = m["ctx"]
    x, y, xd, rb, rc, l2_flush, barrier = c["x"], c["y"], c["xd"], c["rb"], c["rc"], c["l2_flush"], c["barrier"]
    e1d, e2d, radd = c["e1d"], c["e2d"], c["radd"]

    # ---- e2e: the public API with HOST inputs (pinned), H2D + D2H inside the timed region ----
    e2e = None
    if world == 1:
        xh, yh = x.pin_memory(), y.pin_memory()
        xdev = torch.empty_like(xd); ydev = torch.empty(w["n"], device=dev)
        lik = gp.likelihoods.GaussianLikelihood().to(dev)
        lik.noise = w["noise"]
        base = gp.kernels.RBFKernel() if w["kind"] == "rbf" else gp.kernels.MaternKernel(nu={"matern12": 0.5, "matern32": 1.5, "matern52": 2.5}[w["kind"]])
        base.lengthscale = w["lengthscale"]
        if "grid" in w:
            base = gp.kernels.GridInterpolationKernel(base, grid_size=w["grid"], num_dims=w["d"], grid_bounds=[(0.0, 1.0)] * w["d"])
        cov = gp.kernels.ScaleKernel(base).to(dev)
        cov.outputscale = w["outputscale"]
        mean = gp.means.ZeroMean()

        class Model(gp.models.ExactGP):
            def __init__(self):
                super().__init__(xdev, ydev, lik)
                self.mean_module, self.covar_module = mean, cov

            def forward(self, xx):
                return gp.distributions.MultivariateNormal(self.mean_module(xx), self.covar_module(xx))

        model = Model().to(dev)
        mll = gp.mlls.ExactMarginalLogLikelihood(lik, model)
        model.train(); lik.train()

        def e2e_step():
            l2_flush.zero_()
            xdev.copy_(xh, non_blocking=True)   # new inputs arrive from the host: the engine re-packs its tiles
            ydev.copy_(yh, non_blocking=True)
            with torch.no_grad(), settings.max_preconditioner_size(w["rank"]), settings.num_trace_samples(w["probes"]), \
                    settings.backend(args.backend), settings.probe_seed(1):
                out = mll(model(xdev), ydev)
            return float(out.item())  # D2H read of the result

        for _ in range(max(args.warmup, 1)):
            e2e_step()
        torch.cuda.synchronize(dev)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            last = e2e_step()
        f1.record()
        torch.cuda.synchronize(dev)
        ems = f0.elapsed_time(f1) / args.steps
        e2e = {"value": 1e3 / ems, "unit": UNIT, "h2d_bytes_per_step": int(x.numel() * 4 + y.numel() * 4),
               "d2h_bytes_per_step": 4, "ms_per_step": ems,
               "api": "gpytorch_b200.mlls.ExactMarginalLogLikelihood(model(x), y)" + (" with GridInterpolationKernel" if "grid" in w else ""),
               "mll": last}
    else:
        # multi-GPU: same call through the engine API with host inputs on every rank
        xh, yh = x.pin_memory(), y[rb : rb + rc].contiguous().pin_memory()
        xdev = torch.empty_like(xd); ydev = torch.empty(rc, device=dev)
        plan2 = Plan(xdev, backend=args.backend, row_begin=rb, row_count=rc, comm=comm)

        def e2e_step():
            l2_flush.zero_()
            xdev.copy_(xh, non_blocking=True); ydev.copy_(yh, non_blocking=True)
            plan2.refresh_data()
            plan2.set_hypers(w["kind"], w["lengthscale"], w["outputscale"], w["noise"])
            r, _ = plan2.mll(ydev, e1d, e2d, radd, w["probes"], w["rank"], MLL_KNOBS["min_precond_size"], MLL_KNOBS["precond_tol"],
                             MLL_KNOBS["cg_tol"], MLL_KNOBS["max_cg_iter"], MLL_KNOBS["max_tridiag_iter"], warn=False)
            return r.mll

        for _ in range(max(args.warmup, 1)):
            e2e_step()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            last = e2e_step()
        f1.record()
        barrier()
        t2 = torch.tensor([f0.elapsed_time(f1)], device=dev, dtype=torch.float64)
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ems = float(t2.item()) / args.steps
        e2e = {"value": 1e3 / ems, "unit": UNIT, "h2d_bytes_per_step": int(x.numel() * 4 + rc * 4) * world, "d2h_bytes_per_step": 8 * world,
               "ms_per_step": ems, "api": "gpytorch_b200.Plan.mll (row-sharded)", "mll": last}
        plan2.close()

    # ---- secondary record: the 8-GPU strong-scaling configuration (BASELINE configs[2]) on the same ranks, so that the
    # driver's 1/2/4/8 sweep of this script also carries the N=200k curve the north star quotes ----
    c3 = None
    if args.workload == "c2" and not args.no_c3 and WORKLOADS["c3"]["n"] % world == 0:
        c["plan"].close()
        del m["ctx"], c, xd, l2_flush
        torch.cuda.empty_cache()
        w3 = WORKLOADS["c3"]
        m3 = measure_workload(w3, args, env, steps=args.steps, warmup=2)
        c3 = {"metric": METRIC, "value": m3["value"], "unit": UNIT, "ms_per_step": m3["ms_per_step"], "steps": args.steps,
              "warmup": 2, "scaling": "strong", "config": result_config(w3, world, m3),
              "roofline": {k: m3["roofline"][k] for k in ("achieved", "peak", "frac", "ms_per_launch", "mufu_bound")}}
        m3["ctx"]["plan"].close()

    if rank == 0:
        cpu = cpu_baseline(w) if not args.no_cpu else None
        res = m["res"]
        parity = None
        if cpu and cpu.get("value"):
            rel = lambda a, b: abs(a - b) / max(abs(b), 1e-300)  # noqa: E731
            parity = {"against": "cpu_baseline (oracle port, fp32, same inputs and probe base samples, same process)",
                      "cg_iters_equal": bool(res.cg_iters == cpu["cg_iters"]), "inv_quad_rel": rel(res.inv_quad, cpu["inv_quad"]),
                      "logdet_rel": rel(res.logdet, cpu["logdet"]), "mll_abs": abs(res.mll - cpu["mll"])}
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": result_config(w, world, m),
            "clocks": m["clocks"], "e2e": e2e, "gpu_launches": m["launches"], "roofline": m["roofline"], "cpu_baseline": cpu,
            "parity_at_config": parity, "c3": c3,
        }
        emit(line)
        if args.dump_outputs:
            arrays = mll_result_arrays(res, w["probes"] + 1)
            arrays["e2e_mll"] = e2e["mll"]
            if c3:
                arrays.update(mll_result_arrays(m3["res"], w3["probes"] + 1, "c3_"))
            dump_outputs(args.dump_outputs, arrays)
    if world > 1:
        dist.barrier()
        comm.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("GP_WORKLOAD", "c2"), choices=sorted(WORKLOADS))
    ap.add_argument("--backend", default="auto", choices=["auto", "tcgen05", "simt"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-c3", action="store_true", help="skip the secondary N=200k record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (MLL, inv_quad, logdet, ...) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    elif args.workload == "c4":
        run_c4(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
