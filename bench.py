#!/usr/bin/env python
"""bench.py -- the hot-path benchmark (contract: see the task statement / DESIGN.md section 6).

Metric (BASELINE.json): GP log_probability/sec at N=65536, dense ExpSquared 3-D, fp64.
A "step" is one full ``log_probability``: kernel-matrix build fused into the blocked Cholesky,
forward triangular solve, log-determinant and |alpha|^2 reductions.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload dense|quasisep]
                  [--dump-outputs DIR]

* ``value``  : device-timed throughput with X / diag / y already resident in HBM.
* ``e2e``    : the same metric through the public API ``GaussianProcess(kernel, X, diag=...).log_probability(y)``
               with HOST numpy buffers (host->device copies and device->host reads inside the timed region).
* ``roofline``: trailing-update DMMA kernel, algorithmic flop / summed CUDA-event time of its launches,
               against the fp64 tensor (DMMA) peak measured by our own micro-benchmark on this GPU
               (MEASURED_PEAKS.json carries only bf16/HBM peaks; fp64 has no entry there).
* ``cpu_baseline`` / ``--impl reference``: the NumPy/SciPy oracle port (the reference needs JAX, which is not
               installed here or on the box) on the host cores, on a bounded sample, extrapolated as stated.
N > 1: one process per GPU; the dense path runs as independent replicas (one hyper-parameter point per
rank, no data-path collective) -> "scaling": "weak".
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_DENSE = 65536
NDIM = 3
SEED = 49382
OUTPUTS = {}     # name -> what a timed path returned in its last step (written by --dump-outputs)


def make_dense_problem(n, rank=0):
    """SURVEY 8(d) C2: X ~ U(0,20)^3 at N=65536 (same point density for other N), y = sin(x0) + 0.1 N(0,1),
    1.0 * ExpSquared(scale=1.0), diag=0.1.  Ranks > 0 evaluate a neighbouring length scale."""
    rng = np.random.default_rng(SEED)
    side = 20.0 * (n / 65536.0) ** (1.0 / 3.0)
    X = np.ascontiguousarray(rng.uniform(0.0, side, (n, NDIM)))
    y = np.sin(X[:, 0]) + 0.1 * rng.normal(size=n)
    diag = np.full(n, 0.1)
    scale = 1.0 + 0.01 * rank
    return X, y, diag, scale


def golden_check(which, n, logp):
    """full-size LAPACK known answer (tests/golden/full_size.json, made by tests/golden/make_golden_full.py)"""
    try:
        g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden",
                                        "full_size.json")))[which]
    except Exception:
        return None
    if g["n"] != n:
        return None
    return {"log_probability": g["log_probability"], "rel_err": abs(logp - g["log_probability"]) / abs(g["log_probability"]),
            "source": g["lapack"]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(np.min(sm)), "sm_max_mhz": float(np.max(mx)),
                "power_w_median": float(np.median(pw)), "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU oracle leg (cpu_baseline and --impl reference)
# ------------------------------------------------------------------------------------------------
_USED_THREADS = [1]


def oracle_dense_logp_seconds(n):
    """One oracle log_probability on ALL host cores (torchrun exports OMP_NUM_THREADS=1; undo that here).
    Returns (t_build, t_rest, logp): the O(N^2) kernel-matrix build (kernels/base.py:84-103 + noise.py:77-78) and the
    O(N^3) rest (LAPACK dpotrf = direct.py:53, triangular solve, reductions) are timed SEPARATELY so that each can be
    extrapolated with its own exponent."""
    from oracle import tinygp_np as o
    import scipy.linalg as sla
    X, y, diag, scale = make_dense_problem(n)
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        limiter = threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        limiter = None
    try:
        kernel = o.Constant(1.0) * o.ExpSquared(scale)
        noise = o.Diagonal(diag)
        t0 = time.perf_counter()
        K = noise.add_to(kernel(X, X))                                            # direct.py:51
        t1 = time.perf_counter()
        L = sla.cholesky(K, lower=True, check_finite=False, overwrite_a=True)     # direct.py:53
        alpha = sla.solve_triangular(L, y, lower=True, check_finite=False)        # gp.py:320
        lp = -0.5 * np.sum(alpha ** 2) - (np.sum(np.log(np.diag(L))) + 0.5 * n * np.log(2 * np.pi))   # gp.py:313-316
        t2 = time.perf_counter()
        try:
            # the LAPACK / BLAS pool that actually ran dpotrf (not torch's OpenMP pool, which bench.py's own arm also loads)
            blas = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
            _USED_THREADS[0] = max(blas or [p.get("num_threads", 1) for p in threadpool_info()] or [1])
        except Exception:
            pass
    finally:
        if limiter is not None:
            limiter.restore_original_limits()
    return t1 - t0, t2 - t1, float(lp)


def cpu_threads():
    return int(_USED_THREADS[0])


def pick_sample_n(budget_s_per_step):
    """Calibrate on N=4096 and pick the largest sample whose step fits the budget."""
    tb, tr, _ = oracle_dense_logp_seconds(4096)
    for n in (16384, 12288, 8192):
        if tb * (n / 4096.0) ** 2 + tr * (n / 4096.0) ** 3 <= budget_s_per_step:
            return n
    return 8192


def extrapolate(tb, tr, n_s, n):
    """build ~ N^2, factor + solve ~ N^3"""
    return tb * (n / n_s) ** 2 + tr * (n / n_s) ** 3


def full_size_cpu_record():
    """the one full-size CPU run on record (tests/golden/full_size.json, made by tests/golden/make_golden_full.py)"""
    try:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "full_size.json")))["c2"]
        return {"build_s": g.get("build_s"), "factor_s": g.get("dpotrf_s"), "source": g.get("lapack")}
    except Exception:
        return None


def run_reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path: tinygp needs jax + equinox, neither of which is
    installed here or on the GPU box (no network), so this is the NumPy/SciPy/LAPACK oracle port
    (oracle/tinygp_np.py: same formulas, LAPACK dpotrf = what XLA:CPU calls), all host threads, on a bounded sample of
    the workload; the build and the factorisation are extrapolated separately (N^2 / N^3)."""
    if rank != 0:
        return
    np.random.seed(0)
    total_budget = 150.0
    n_s = pick_sample_n(total_budget / max(1, args.steps + args.warmup))
    for _ in range(args.warmup):
        oracle_dense_logp_seconds(n_s)
    tbs, trs = [], []
    for _ in range(args.steps):
        tb, tr, lp = oracle_dense_logp_seconds(n_s)
        tbs.append(tb); trs.append(tr)
    tb, tr = float(np.median(tbs)), float(np.median(trs))
    t_full = extrapolate(tb, tr, n_s, N_DENSE)
    value = 1.0 / t_full
    cores = cpu_threads()
    sample = (f"N={n_s} of the same workload per step: build {tb:.2f} s (x{(N_DENSE / n_s) ** 2:.0f}, N^2) + "
              f"dpotrf/solve {tr:.2f} s (x{(N_DENSE / n_s) ** 3:.0f}, N^3) -> {t_full:.0f} s at N={N_DENSE}")
    line = {
        "impl": "reference", "metric": "log_probability/sec", "value": value, "unit": "logp/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_full * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"dense ExpSquared 3-D N={N_DENSE} log_probability (build + Cholesky + solve)",
                   "kernel": "1.0*ExpSquared(scale=1.0), L2", "diag": 0.1, "seed": SEED,
                   "same_config": False, "note": "oracle port on a bounded sample, extrapolated (see cpu_baseline.sample)"},
        "cpu_baseline": {"value": value, "unit": "logp/s", "cores": cores, "kind": "port", "sample": sample,
                         "full_size_run_on_record": full_size_cpu_record()},
        "e2e": {"value": value, "unit": "logp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "per_step_s_at_sample": [round(a + b, 3) for a, b in zip(tbs, trs)],
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    from tinygp_b200 import GaussianProcess, _cabi, kernels

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device visible; the B200 solver has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from tinygp_b200 import multigpu
    ctx = multigpu.make_context(local_rank)      # library + torch share one (non-default) CUDA stream
    stream = torch.cuda.current_stream()
    ctx.set_option("nb", args.nb)
    ctx.set_option("ozaki_slices", args.slices)
    ctx.set_option("ozaki_min_n", 0 if args.slices else 1 << 40)
    for kv in args.opt:                            # tuning experiments: --opt ozaki_pairing=1 --opt ozaki_layout=1 ...
        key, _, val = kv.partition("=")
        ctx.set_option(key, int(val))

    n = args.n
    X, y, diag, scale = make_dense_problem(n, rank)
    kernel = 1.0 * kernels.ExpSquared(scale=scale)
    prog = kernel.program()
    from ctypes import byref, c_double
    dX = torch.from_numpy(X).cuda()
    dy = torch.from_numpy(y).cuda()
    ddiag = torch.from_numpy(diag).cuda()
    lp = c_double()

    def step_device():
        ctx.check(ctx.lib.b200gp_dense_log_probability_dev(
            ctx.handle, _cabi.ptr(prog), prog.shape[0], dX.data_ptr(), n, NDIM, ddiag.data_ptr(), dy.data_ptr(),
            byref(lp)))
        return lp.value

    # e2e inputs in pinned host memory (NumPy views of page-locked torch tensors; the host layer passes them through)
    Xp, yp, diagp = (torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in (X, y, diag))

    def step_e2e():
        return GaussianProcess(kernel, Xp, diag=diagp).log_probability(yp)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_step_ms = []

    def timed(fn, steps, record=None):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        evs[0].record(stream)
        out = None
        for i in range(steps):
            out = fn()
            evs[i + 1].record(stream)
        barrier()
        if record is not None:
            record.extend(round(evs[i].elapsed_time(evs[i + 1]), 3) for i in range(steps))
        from tinygp_b200.parallel import max_over_ranks
        return max_over_ranks(evs[0].elapsed_time(evs[steps]), device="cuda"), out

    # fp64 tensor peak on this GPU: burst (short loop) and sustained (~2 s loop, the denominator for a kernel
    # timed inside a multi-second step)
    peak_burst = max(ctx.measure_fp64_peak()[0] for _ in range(3))
    ctx.set_option("peak_iters", 1_500_000)
    peak_sustained, dfma_sustained = ctx.measure_fp64_peak()
    ctx.set_option("peak_iters", 4096)
    i8_peak_burst = max(ctx.measure_i8_peak() for _ in range(2))
    ctx.set_option("peak_iters", 200000)
    i8_peak_sustained = ctx.measure_i8_peak()
    ctx.set_option("peak_iters", 4096)

    for _ in range(args.warmup):
        step_device()
    l0 = ctx.launch_count()
    ctx.set_option("profile", 1)
    ctx.profile(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, logp = timed(step_device, args.steps, per_step_ms)
    OUTPUTS["log_probability"] = logp
    clocks = sampler.stop() if rank == 0 else None
    prof = ctx.profile(reset=True)
    ctx.set_option("profile", 0)
    launches = ctx.launch_count() - l0

    # e2e through the public API with host buffers
    e2e_steps = args.steps
    if args.quick:                       # tuning sweeps only: the line is then NOT a valid bench line (no e2e, no baseline)
        ms_e2e, logp_e2e = float("nan"), float("nan")
    else:
        step_e2e()
        ms_e2e, logp_e2e = timed(step_e2e, e2e_steps)
        OUTPUTS["log_probability_e2e"] = logp_e2e

    # ---- the other BASELINE configs, attached to the one line the driver parses --------------------------------------
    sub_records, sharded = {}, None
    if not args.quick and not args.no_sub:
        ctx.set_option("trim", 0)            # give the cached 34 GB matrix + digit planes back before the next workloads
        if world > 1:
            # BASELINE config 3: ONE factorisation sharded over all ranks (collective: every rank takes part)
            try:
                sharded = measure_sharded(args, ctx, rank, local_rank, world, warmup=1)
            except Exception as e:  # noqa: BLE001
                sharded = {"error": str(e)[:300]}
        elif rank == 0:
            for name, fn in (("c4_quasisep", measure_quasisep), ("c5_batched", measure_batched)):
                try:
                    ctx.reset_options()
                    sub_records[name] = fn(args, ctx, local_rank)
                except Exception as e:  # noqa: BLE001
                    sub_records[name] = {"error": str(e)[:300]}
                ctx.set_option("trim", 0)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * args.steps / (ms * 1e-3)
    e2e_value = world * e2e_steps / (ms_e2e * 1e-3)
    flop_alg = n ** 3 / 3.0
    syrk_tf = prof["syrk_flop"] / max(prof["syrk_ms"], 1e-9) / 1e9
    if args.slices:
        i8_tops = prof["i8_ops"] / max(prof["syrk_ms"], 1e-9) / 1e9
        try:
            bf16 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            bf16 = {}
        roofline = {
            "bound": "tensor", "kernel": "i8_update_kernel (tcgen05.mma kind::i8, TMA multicast, TMEM int32 accumulators)",
            "achieved": i8_tops, "peak": i8_peak_sustained, "unit": "TFLOP/s", "frac": i8_tops / i8_peak_sustained,
            "peak_source": "int8 tensor TOP/s measured on this GPU by b200gp_measure_i8_peak (resident-operand "
                           "tcgen05 loop, ~1 s); MEASURED_PEAKS.json has bf16 only (int8 nominal = 2x bf16)",
            "peak_burst": i8_peak_burst, "bf16_measured_peaks": {k: bf16.get(k) for k in ("bf16_tflops", "bf16_tflops_sustained")},
            "int8_ops_per_step": prof["i8_ops"] / args.steps, "digit_planes": args.slices,
            "fp64_equivalent_tflops": syrk_tf, "fp64_dmma_peak_sustained": peak_sustained, "fp64_dmma_peak_burst": peak_burst,
            "launches": int(prof["syrk_launches"]), "ms_total": prof["syrk_ms"],
            "whole_step_tflops_n3_over_3": flop_alg * args.steps / (ms * 1e-3) / 1e12,
            "traffic": _read_traffic(),
        }
    else:
      roofline = {
        "bound": "tensor", "kernel": "gemm_nt_kernel<true> (trailing SYRK/GEMM update, DMMA m8n8k4 f64)",
        "achieved": syrk_tf, "peak": peak_sustained, "unit": "TFLOP/s", "frac": syrk_tf / peak_sustained,
        "peak_source": "measured on this GPU by b200gp_measure_fp64_peak (sustained ~2 s DMMA loop); "
                       "MEASURED_PEAKS.json has no fp64 entry",
        "peak_burst": peak_burst, "dfma_sustained": dfma_sustained,
        "launches": int(prof["syrk_launches"]), "ms_total": prof["syrk_ms"],
        "whole_step_tflops_n3_over_3": flop_alg * args.steps / (ms * 1e-3) / 1e12,
        "traffic": _read_traffic(),
      }
    # CPU baseline on a bounded sample (rank 0 at N=1 only)
    if world == 1 and not args.quick:
        n_s = pick_sample_n(25.0)
        tb, tr, lp_cpu = oracle_dense_logp_seconds(n_s)
        t_full = extrapolate(tb, tr, n_s, n)
        cpu_baseline = {"value": 1.0 / t_full, "unit": "logp/s", "cores": cpu_threads(), "kind": "port",
                        "sample": f"N={n_s} timed: build {tb:.2f} s (x{(n / n_s) ** 2:.0f}, N^2) + dpotrf/solve {tr:.2f} s "
                                  f"(x{(n / n_s) ** 3:.0f}, N^3) -> {t_full:.0f} s at N={n}",
                        "full_size_run_on_record": full_size_cpu_record()}
    else:
        cpu_baseline = None

    line = {
        "metric": "log_probability/sec", "value": value, "unit": "logp/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"dense ExpSquared 3-D N={n} log_probability (fused build + blocked Cholesky + solve)",
                   "kernel": "1.0*ExpSquared(scale=1.0), L2", "diag": 0.1, "seed": SEED, "nb": args.nb,
                   "trailing_update": (f"int8 fixed-point, {args.slices} digit planes (tcgen05 kind::i8)" if args.slices
                                       else "native fp64 DMMA"),
                   "options": args.opt, "quick": bool(args.quick),
                   "parallelism": f"replicas x{world}" if world > 1 else "single GPU",
                   "l2": "working set 34 GB >> 126 MB L2 (no flush needed)"},
        "logp": logp, "logp_e2e": logp_e2e, "golden": golden_check("c2", n, logp),
        "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "logp/s", "steps": e2e_steps,
                "h2d_bytes_per_step": int(n * NDIM * 8 + n * 8 + n * 8),
                "d2h_bytes_per_step": int(n * 8 + n * 8 + 8 + 4)},
        "gpu_launches": int(launches),
        "kernel_ms_per_step": {"syrk": prof["syrk_ms"] / args.steps, "panel": prof["panel_ms"] / args.steps,
                               "build": prof["build_ms"] / args.steps},
        "per_step_ms": per_step_ms,
    }
    # the forward substitution: a serial phase of its own (13 ms at N = 65536), or -- option solve_overlap, default -- launches
    # on a side stream that are IN FLIGHT under the int8 update of the next block column (event time = residence, not cost)
    solve_key = "solve_in_flight_under_update" if (args.slices > 0 and ctx.get_option("solve_overlap")) else "solve"
    line["kernel_ms_per_step"][solve_key] = prof["solve_ms"] / args.steps
    if sub_records:
        line["configs"] = sub_records
    if sharded is not None:
        line["sharded"] = sharded
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _hbm_peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def measure_quasisep(args, ctx, local_rank, n=10_000_000, warmup=3, opts=()):
    """BASELINE config 4: SHO + Matern-3/2 (J = 4) on a sorted 1-D series of N = 1e7 points, one GPU.
    `value`: device-resident inputs through b200gp_qs_log_probability_dev; `e2e`: GaussianProcess(...).log_probability(y)
    with host buffers.  The C restatement of the sequential recursion (oracle/csrc) checks the FULL series."""
    import torch
    from ctypes import byref, c_double, c_int
    from tinygp_b200 import GaussianProcess, _cabi
    from tinygp_b200.kernels import quasisep as Q

    steps = args.steps
    stream = torch.cuda.current_stream()
    for kv in opts:
        key, _, val = kv.partition("=")
        ctx.set_option(key, int(val))
    rng = np.random.default_rng(49384)
    t = np.sort(rng.uniform(0, n / 10.0, n))
    y = np.sin(t) + 0.1 * rng.normal(size=n)
    diag = np.full(n, 0.1)
    kernel = Q.SHO(omega=1.5, quality=3.0, sigma=1.8) + Q.Matern32(scale=1.5, sigma=0.9)
    comps = kernel.component_array()
    dt, dy, dd = (torch.from_numpy(a).cuda() for a in (t, y, diag))
    lp, uns = c_double(), c_int()

    def step_device():
        ctx.check(ctx.lib.b200gp_qs_log_probability_dev(ctx.handle, _cabi.ptr(comps), comps.shape[0], dt.data_ptr(), n,
                                                        dd.data_ptr(), dy.data_ptr(), 1, byref(uns), byref(lp)))
        return lp.value

    # e2e: host buffers in PINNED memory (the contract's "from pinned host memory"): NumPy views of page-locked torch tensors,
    # which the host layer passes through unchanged (already C-contiguous float64), so the library's cudaMemcpyAsync runs at
    # PCIe rate instead of through the driver's pageable staging
    tp, yp, dp = (torch.from_numpy(a).pin_memory().numpy() for a in (t, y, diag))

    def step_e2e():
        return GaussianProcess(kernel, tp, diag=dp, assume_sorted=True).log_probability(yp)

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(k):
            out = fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(warmup):
        step_device()
    ctx.set_option("profile", 1)
    ctx.profile(reset=True)
    l0 = ctx.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, logp = timed(step_device, steps)
    clocks = sampler.stop()
    prof = ctx.profile(reset=True)
    ctx.set_option("profile", 0)
    launches = ctx.launch_count() - l0
    step_e2e()
    e2e_steps = steps
    ms_e2e, logp_e2e = timed(step_e2e, e2e_steps)
    OUTPUTS.update(quasisep_log_probability=logp, quasisep_log_probability_e2e=logp_e2e)
    J = kernel.state_dim()
    alg_bytes = 8.0 * n * (3 + 1 + J)          # read t, diag, y ; write c, w   (SURVEY 8d: 64 B/point at J=4)
    hbm_peak, src = _hbm_peak()
    achieved = alg_bytes * steps / (prof["qs_ms"] * 1e-3) / 1e9
    # parity at FULL size: the C restatement of ops.py:352-365,463-472 on all N points (1 core)
    from oracle import cref, tinygp_np as o
    ko = o.qs.SHO(1.5, 3.0, 1.8) + o.qs.Matern32(1.5, 0.9)
    d_, p_, q_, a_ = o.qs_generators_fast(ko, t)
    t0 = time.perf_counter()
    lpo = cref.qs_log_probability(d_ + 0.1, p_, q_, a_, y)
    t_cpu = time.perf_counter() - t0
    del d_, p_, q_, a_
    return {
        "metric": "log_probability/sec", "value": steps / (ms * 1e-3), "unit": "logp/s", "n_gpus": 1,
        "steps": steps, "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"quasisep SHO+Matern32 (J=4) N={n} log_probability", "diag": 0.1, "seed": 49384,
                   "options": list(opts), "l2": "working set 0.64 GB > 126 MB L2"},
        "logp": logp, "logp_e2e": logp_e2e,
        "parity": {"oracle_logp": lpo, "rel_err": abs(logp - lpo) / abs(lpo), "rel_err_e2e": abs(logp_e2e - lpo) / abs(lpo),
                   "oracle": f"C restatement of the sequential recursion on all {n} points ({t_cpu:.2f} s, 1 core)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                     "peak_source": src, "traffic": _read_traffic("qs_traffic.json", "dram_bytes_per_step") if n == 10_000_000 else None,
                     "algorithmic_bytes_per_point": 8 * (3 + 1 + J),
                     "note": "fp64-ALU bound (Riccati composites + exp/sincos per point), see DESIGN.md section 4"},
        "cpu_baseline": {"value": 1.0 / t_cpu, "unit": "logp/s", "cores": 1, "kind": "port",
                         "sample": f"all {n} points, C restatement of ops.py:352-365,463-472 ({t_cpu:.2f} s; generators "
                                   f"precomputed with NumPy, not timed)"},
        "clocks": clocks,
        "e2e": {"value": e2e_steps / (ms_e2e * 1e-3), "unit": "logp/s", "h2d_bytes_per_step": int(3 * 8 * n),
                "d2h_bytes_per_step": 16,
                "note": "pinned host buffers; 240 MB over PCIe per call (t, diag, y) bound e2e at ~200 logp/s whatever the kernels do"},
        "gpu_launches": int(launches), "kernel_ms_per_step": {"qs": prof["qs_ms"] / steps},
    }


def run_quasisep(args, rank, local_rank, world):
    """BASELINE config 4 as a stand-alone workload (python bench.py --workload quasisep)."""
    from tinygp_b200 import multigpu
    ctx = multigpu.make_context(local_rank)
    if args.qs_chunk:
        ctx.set_option("qs_chunk", args.qs_chunk)
    n = args.n if args.n != N_DENSE else 10_000_000
    line = measure_quasisep(args, ctx, local_rank, n=n, warmup=args.warmup, opts=args.opt)
    line.update({"scaling": "weak", "vs_baseline": None})
    print(json.dumps(line), flush=True)


def measure_batched(args, ctx, local_rank, rank=0, world=1, n=4096, warmup=1):
    """BASELINE config 5: 1024 independent N=4096 ExpSquared problems (32 x 32 hyper-parameter grid), sharded
    128 per GPU at 8 GPUs -- replicas only, no data-path collective."""
    import torch
    import torch.distributed as dist
    from tinygp_b200 import _cabi, kernels

    stream = torch.cuda.current_stream()
    steps = args.steps
    nprob = 1024
    rng = np.random.default_rng(49385)
    X = np.ascontiguousarray(rng.uniform(0, 8, (n, 3)))
    y = np.sin(X[:, 0]) + 0.1 * rng.normal(size=n)
    diag = np.full(n, 0.1)
    grid = [(sc, a) for sc in np.logspace(-0.5, 0.5, 32) for a in np.logspace(-1, 1, 32)]
    from tinygp_b200.parallel import shard_indices
    mine = [grid[i] for i in shard_indices(len(grid), rank, world)]
    progs = np.ascontiguousarray(np.stack([(a * kernels.ExpSquared(scale=sc)).program() for sc, a in mine]))
    out = np.empty(len(mine))

    def step():
        ctx.check(ctx.lib.b200gp_dense_log_probability_batched(
            ctx.handle, _cabi.ptr(progs), progs.shape[1], len(mine), _cabi.ptr(X), n, 3, _cabi.ptr(diag), _cabi.ptr(y),
            _cabi.ptr(out)))

    for _ in range(warmup):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    t = float(ms.item()) * 1e-3
    OUTPUTS["batched_log_probability"] = out.copy()
    # parity on the corners of the grid this rank holds (oracle: LAPACK at N = 4096, ~1 s each)
    from oracle import tinygp_np as o
    checks = []
    if rank == 0:
        for idx in (0, len(mine) - 1):
            sc, a = mine[idx]
            lpo = o.GaussianProcess(o.Constant(a) * o.ExpSquared(sc), X, diag=0.1).log_probability(y)
            checks.append(abs(out[idx] - lpo) / abs(lpo))
    tf = nprob * steps * n ** 3 / 3 / t / 1e12
    return {
        "metric": "log_probability/sec", "value": nprob * steps / t, "unit": "logp/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": t * 1e3 / steps, "higher_is_better": True,
        "scaling": "strong", "dtype": "f64", "data": "synthetic", "vs_baseline": None,
        "config": {"workload": f"batched: {nprob} x (N={n}) ExpSquared log_probability, hyper-parameter grid, "
                               f"{len(mine)} problems per GPU (host buffers, end to end)"},
        "tflops_n3_over_3": tf,
        "roofline": {"bound": "tensor", "achieved": tf, "unit": "TFLOP/s", "peak": None,
                     "note": "native fp64 DMMA path (N = 4096 < ozaki_min_n); DMMA peak measured by the dense line"},
        "parity": {"max_rel_err_vs_oracle_on_grid_corners": max(checks) if checks else None},
        "logp_first": float(out[0]), "clocks": clocks,
    }


def run_batched(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from tinygp_b200 import multigpu
    ctx = multigpu.make_context(local_rank)
    n = 4096 if args.n == N_DENSE else args.n
    for kv in args.opt:                            # tuning experiments: --opt nb_batched=1024 ...
        key, _, val = kv.partition("=")
        ctx.set_option(key, int(val))
    line = measure_batched(args, ctx, local_rank, rank, world, n=n, warmup=args.warmup)
    if args.opt:
        line["config"]["options"] = list(args.opt)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_sharded(args, ctx, rank, local_rank, world, n=131072, warmup=1, slices=None):
    """BASELINE config 3: ONE dense log_probability sharded over the GPUs.  Kernel 1.5*Matern52(2.0) +
    0.7*RationalQuadratic(1.5, alpha=1.5), both with the Euclidean metric (the L1 defaults are indefinite in 3-D, see
    DESIGN.md section 2), N = 131072 by default.  Strong scaling.  Collective: every rank must call this."""
    import torch
    import torch.distributed as dist
    from tinygp_b200 import kernels, multigpu

    ctx.set_option("nb", args.nb)
    steps = args.steps
    rng = np.random.default_rng(49383)
    side = 25.0 * (n / 131072.0) ** (1.0 / 3.0)
    X = np.ascontiguousarray(rng.uniform(0.0, side, (n, NDIM)))
    y = np.sin(X[:, 0]) + 0.1 * rng.normal(size=n)
    diag = np.full(n, 0.1)
    L2 = kernels.L2Distance()
    kernel = 1.5 * kernels.Matern52(2.0, L2) + 0.7 * kernels.RationalQuadratic(1.5, L2, alpha=1.5)
    dX, dy, dd = (torch.from_numpy(a).cuda() for a in (X, y, diag))
    slices = slices or args.slices or 7
    stats = {}

    def step():
        return multigpu.log_probability_sharded(kernel, None, None, None, slices=slices, ctx=ctx, X_dev=dX, diag_dev=dd,
                                                resid_dev=dy, stats=stats)

    from tinygp_b200.parallel import max_over_ranks
    for _ in range(warmup):
        step()
    stream = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ctx.set_option("profile", 1)
    ctx.profile(reset=True)
    if rank == 0:
        sampler.start()
    stats.clear()
    e0.record(stream)
    for _ in range(steps):
        lp = step()
    e1.record(stream)
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    prof = ctx.profile(reset=True)
    ctx.set_option("profile", 0)
    ms = max_over_ranks(e0.elapsed_time(e1), device="cuda")
    t = ms * 1e-3
    OUTPUTS["sharded_log_probability"] = lp
    line = {
        "metric": "log_probability/sec", "value": steps / t, "unit": "logp/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"dense Matern52+RationalQuadratic (L2) 3-D N={n}: ONE log_probability sharded over "
                               f"{world} GPU(s), int8 fixed-point update ({slices} digit planes)",
                   "diag": 0.1, "seed": 49383, "nb": args.nb, "exchange": stats.get("exchange", "all_gather_into_tensor per block column")},
        "logp": lp, "golden": golden_check("c3", n, lp) or golden_check("c3s", n, lp),
        "tflops_n3_over_3": n ** 3 / 3.0 * steps / t / 1e12,
        "kernel_ms_per_step_rank0": {"i8_update": prof["syrk_ms"] / steps, "panel": prof["panel_ms"] / steps,
                                     "build_cut": prof["build_ms"] / steps, "solve": prof["solve_ms"] / steps},
        "exchange_bytes_per_step_per_rank": (stats["bytes"] // max(1, steps)) if stats.get("bytes") else 0,
        "clocks": clocks,
    }
    if n <= 16384 and rank == 0:
        from oracle import tinygp_np as o
        ko = o.Constant(1.5) * o.Matern52(2.0, o.L2Distance()) + o.Constant(0.7) * o.RationalQuadratic(
            1.5, o.L2Distance(), alpha=1.5)
        lpo = o.GaussianProcess(ko, X, diag=0.1).log_probability(y)
        line["oracle_logp"] = lpo
        line["rel_err"] = abs(lp - lpo) / abs(lpo)
    return line


def run_sharded(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from tinygp_b200 import multigpu
    ctx = multigpu.make_context(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    for kv in args.opt:
        key, _, val = kv.partition("=")
        ctx.set_option(key, int(val))
    n = 131072 if args.n == N_DENSE else args.n
    line = measure_sharded(args, ctx, rank, local_rank, world, n=n, warmup=args.warmup)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _read_traffic(name="syrk_traffic.json", key="dram_bytes_per_launch"):
    """DRAM read + write bytes of the dominant kernel(s) from the committed ncu capture (profiles/): per launch for the int8
    update, per step for the two point-wise quasiseparable passes"""
    p = os.path.join(ROOT, "profiles", name)
    try:
        return json.load(open(p)).get(key)
    except Exception:
        return None


def dump_outputs(directory):
    """OUTPUTS as DIR/<name>.npy in float64: with the same arguments the inputs are the same seeded arrays, so two builds
    can be compared output for output"""
    os.makedirs(directory, exist_ok=True)
    for name, value in OUTPUTS.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.asarray(value, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed steps of every timed leg: the device path, e2e, and the attached configs")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", "--n", dest="n", type=int, default=N_DENSE, help="problem size N (use --size under torchrun)")
    ap.add_argument("--nb", type=int, default=1024)
    ap.add_argument("--qs-chunk", type=int, default=0)
    ap.add_argument("--workload", default="dense", choices=["dense", "quasisep", "batched", "sharded"])
    ap.add_argument("--slices", type=int, default=7,
                    help="int8 digit planes of the fixed-point trailing update: 7 = 48 bits under the row scale (default: "
                         "same 4.7e-12 distance to the LAPACK golden at N=65536 as 8 planes), 8 = 55 bits, "
                         "0 = native fp64 DMMA")
    ap.add_argument("--quick", action="store_true",
                    help="tuning sweeps: skip the e2e and cpu_baseline legs (the printed line is not a valid bench line)")
    ap.add_argument("--no-sub", action="store_true",
                    help="dense workload: skip the attached sub-records (C4 quasisep, C5 batched; sharded C3 when WORLD_SIZE > 1)")
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=INT",
                    help="library option for tuning runs (b200gp_set_option); dense and quasisep workloads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what each timed path returned in its last step as "
                         "DIR/<name>.npy (float64); rank 0's values (its shard of the batched grid); impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a smaller sample of the workload, not the same outputs")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    elif args.workload == "sharded":
        run_sharded(args, rank, local_rank, world)
    elif args.workload == "batched":
        run_batched(args, rank, local_rank, world)
    elif args.workload == "quasisep":
        if rank == 0:
            run_quasisep(args, rank, local_rank, world)
    else:
        run_ours(args, rank, local_rank, world)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs)


if __name__ == "__main__":
    main()
