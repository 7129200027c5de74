#!/usr/bin/env python
"""Throughput benchmark of the many-chain NUTS hot path (BASELINE.json metric: leapfrog gradient evals/s and
NUTS ESS/s, whole box).

Default workload: BASELINE.json configs[4] ("c5") -- chain-sharded NUTS Bayesian logistic regression, N = 100k,
D = 128, 131072 chains per GPU (1M chains on 8 GPUs), float32 state, gradient on the fused tcgen05 / TMA / TMEM
kernel.  A "step" is TICKS engine ticks in free-running mode; every tick is one velocity-Verlet step (one gradient
evaluation) of every chain, chains finishing and restarting NUTS transitions independently.  At N = 1 the same JSON
line carries the other BASELINE configurations as `secondary`: c3 (configs[2], 4096 chains), c2 (configs[1], d = 1000
dense metric, float64), c4 (configs[3], window adaptation + NUTS on the funnel / eight schools, 65536 chains) and c1
(configs[0], HMC on a 100-dim Gaussian), each with its own value / ms / roofline.

N > 1: chains are sharded (Philox keyed by global chain id), no data-path collective ("weak" scaling).  The
collectives are the adaptation-statistic exchange of the pooled warm-up and the diagnostics exchange (all-gather of
the sorted monitored draws for the rank normalisation, all-reduce of the ESS / R-hat sufficient statistics); both are
inside the timed `e2e_with_diagnostics` number.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c5|c3|c2|c3small|c2small]
                  [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed engine call returned (positions, momenta, energies, gradients, acceptance
statistics, tree depths, flags, leapfrog counts, counters) as DIR/<name>.npy, so that two builds run with the same arguments
-- hence the same seeded inputs -- can be compared output for output (see last_step_outputs).
"""
import argparse
import json
import math
import multiprocessing as mp
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (kind, chains per GPU, dim, ticks per step, data rows)
    "c5": ("logistic", 131072, 128, 32, 100000),
    "c3": ("logistic", 4096, 128, 48, 100000),
    "c2": ("dense", 4096, 1000, 48, 0),
    "c2small": ("dense", 512, 256, 8, 0),
    "c3small": ("logistic", 512, 64, 8, 4096),
}
EPS = {"dense": 0.25, "logistic": 0.4}
METRIC = "leapfrog_gradient_evals_per_sec"
UNIT = "gradient evals/s"
MIN_TIMED_S = 2.0          # secondary workloads choose their step count so that the timed region lasts this long
DUMP_BYTES = 64 * 10 ** 6  # --dump-outputs: all files together stay within this
DUMP_ROW_BYTES = 48 << 20  # ... of which the three [chains, dim] arrays take at most this (a seeded sample of the chains)


# ----------------------------------------------------------------------------------------------------------
# synthetic problems (SURVEY.md 8d); NumPy only, shared by the GPU arm and the CPU arm
# ----------------------------------------------------------------------------------------------------------
def make_dense_problem(d):
    """config 2: Sigma = A A^T / d + 0.1 I (seed 3), Lambda = Sigma^-1, imm = Sigma."""
    rng = np.random.default_rng(3)
    A = rng.standard_normal((d, d))
    cov = A @ A.T / d + 0.1 * np.eye(d)
    prec = np.linalg.inv(cov)
    prec = 0.5 * (prec + prec.T)
    return cov, prec


def bf16_round(x):
    """Round float32 values to the nearest bf16-representable value (ties to even), in NumPy."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.view(np.float32)


def make_logistic_problem(n, d):
    """configs 3/5: X ~ N(0,1) rounded to bf16 (seed 4), beta* ~ N(0,1)/sqrt(D), y ~ Bernoulli(sigmoid(X beta*)),
    prior scale 1, diagonal imm = 4/N."""
    rng = np.random.default_rng(4)
    X = bf16_round(rng.standard_normal((n, d)).astype(np.float32)).astype(np.float64)
    beta = rng.standard_normal(d) / np.sqrt(d)
    y = (rng.random(n) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    return X, y, np.full(d, 4.0 / n)


def make_c1_problem():
    """config 0: mu = 0, sigma_i = exp(N(0, 0.5^2)) (seed 1), imm = sigma^2, HMC L = 10, eps = 0.25."""
    d = 100
    sigma = np.exp(0.5 * np.random.default_rng(1).standard_normal(d))
    return d, sigma


def initial_positions(kind, C, d, chain_offset=0):
    if kind == "dense":
        return np.random.default_rng([5, chain_offset]).standard_normal((C, d))
    return 0.1 * np.random.default_rng([6, chain_offset]).standard_normal((C, d))


def describe(name):
    kind, Cn, d, ticks, n = WORKLOADS[name]
    if kind == "dense":
        which = " (BASELINE.json configs[1])" if name == "c2" else ""
        return f"{name}: NUTS, {d}-dim correlated Gaussian, dense inverse mass matrix, {Cn} chains per GPU{which}"
    which = {"c3": " (BASELINE.json configs[2])", "c5": " (BASELINE.json configs[4]: 1M chains on 8 GPUs)"}.get(name, "")
    return (f"{name}: NUTS, Bayesian logistic regression N={n} D={d}, diagonal inverse mass matrix, "
            f"{Cn} chains per GPU{which}")


def host_ess(draws):
    """bulk-ESS (arviz default: split, rank-normalised) of host draws [T, C, d'], min over dims; NumPy/torch-CPU."""
    import torch
    from aehmc_b200 import diagnostics
    if draws.shape[0] < 4:
        return None
    return float(np.nanmin(diagnostics.ess(torch.from_numpy(np.ascontiguousarray(draws)), distributed=False)))


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (NumPy restatement of the reference, one chain per process, 1 BLAS thread each)
# ----------------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    name, n_transitions, seed = args
    try:
        from threadpoolctl import threadpool_limits
        limiter = threadpool_limits(limits=1)
    except Exception:
        limiter = None
    from oracle import kernels, models, streams
    kind, _, d, _, n = WORKLOADS[name]
    if kind == "dense":
        cov, prec = make_dense_problem(d)
        model, imm = models.CorrelatedGaussian(np.zeros(d), prec), cov
    else:
        X, y, imm = make_logistic_problem(n, d)
        model = models.LogisticRegression(X, y, 1.0)
    srng = streams.StreamDraws(seed, "nuts")
    kernel = kernels.nuts_new_kernel(srng, model)
    q0 = initial_positions(kind, 1, d, seed)[0]
    state = kernels.new_state(q0, model)
    n_leap, pos, acc = 0, [], []
    t0 = time.perf_counter()
    for _ in range(n_transitions):
        info, extras = kernel(state, EPS[kind], imm)
        n_leap += extras["n_leapfrog"]
        pos.append(np.asarray(info.state.position)[:8].copy())
        acc.append(float(info.acceptance_probability))
        state = info.state._replace(momentum=None)
    dt = time.perf_counter() - t0
    del limiter
    return n_leap, dt, np.array(pos), float(np.mean(acc))


def cpu_transitions(name, n_samples=1):
    """NUTS transitions per oracle chain in one CPU sample; shrunk when many samples are requested so that the
    whole reference arm stays within a few minutes (about 0.3 s per c2 transition, 0.2 s per c3 transition)."""
    kind, _, d, _, n = WORKLOADS[name]
    if kind == "dense":
        full = 30 if d >= 1000 else 60
        return max(4, min(full, (8 * full) // max(n_samples, 1)))
    full = 20 if n >= 100000 else 60
    return max(3, min(full, (8 * full) // max(n_samples, 1)))


def cpu_reference_sample(name, cores, n_transitions):
    """All host cores, one oracle chain each; returns a dict (evals/s aggregate, leapfrogs, wall seconds, ESS/s)."""
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(name, n_transitions, 1000 + i) for i in range(cores)])
    wall = time.perf_counter() - t0
    n_leap = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    draws = np.stack([r[2] for r in res], axis=1)                    # [T, cores, 8]
    ess = host_ess(draws)
    return {"value": n_leap / busy, "leapfrogs": n_leap, "wall_s": wall, "busy_s": busy,
            "ess_per_sec": None if ess is None else ess / busy, "mean_accept": float(np.mean([r[3] for r in res]))}


def cpu_c1_sample(n_transitions=1000, burn=100):
    """configs[0] as the reference runs it: ONE chain, single-threaded (OMP_NUM_THREADS=1 in the reference's CI),
    HMC velocity_verlet L = 10, diagonal inverse mass matrix, 100-dim iid Gaussian."""
    try:
        from threadpoolctl import threadpool_limits
        limiter = threadpool_limits(limits=1)
    except Exception:
        limiter = None
    from oracle import kernels, models, streams
    d, sigma = make_c1_problem()
    model = models.IIDGaussian(np.zeros(d), sigma)
    kernel = kernels.hmc_new_kernel(streams.StreamDraws(11, "hmc"), model)
    state = kernels.new_state(np.random.default_rng(2).standard_normal(d), model)
    L, eps, imm = 10, 0.25, sigma ** 2
    pos, acc = [], []
    for i in range(burn + n_transitions):
        if i == burn:
            t0 = time.perf_counter()
        info, _ = kernel(state, eps, imm, L)
        state = info.state._replace(momentum=None)
        if i >= burn:
            pos.append(np.asarray(info.state.position)[:8].copy())
            acc.append(float(info.acceptance_probability))
    dt = time.perf_counter() - t0
    del limiter
    ess = host_ess(np.array(pos)[:, None, :])
    return {"value": n_transitions * L / dt, "unit": UNIT, "cores": 1, "kind": "port", "seconds": dt,
            "ess_per_sec": None if ess is None else ess / dt, "mean_accept": float(np.mean(acc)),
            "sample": f"1 oracle chain, {burn} burn-in + {n_transitions} HMC transitions of L = {L}, single-threaded"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, _, d, _, n = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    warm = min(args.warmup, 1)
    n_tr = cpu_transitions(args.workload, warm + args.steps)
    vals = []
    for i in range(warm + args.steps):
        r = cpu_reference_sample(args.workload, cores, n_tr)
        if i >= warm:
            vals.append(r)
    value = float(np.mean([v["value"] for v in vals]))
    ms = float(np.mean([v["wall_s"] for v in vals]) * 1e3)
    ess = [v["ess_per_sec"] for v in vals if v["ess_per_sec"] is not None]
    sample = (f"{cores} oracle chains (one per core, 1 BLAS thread each) x {n_tr} NUTS transitions of the "
              f"{args.workload} target per step")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": describe(args.workload) + " -- CPU arm: NumPy oracle restating aesara-devs/aehmc "
                               "(the real reference needs Aesara, which is not installable here)",
                   "chains": cores, "dim": d, "step_size": EPS[kind],
                   "mean_accept": float(np.mean([v["mean_accept"] for v in vals]))},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "ess_per_sec": float(np.mean(ess)) if ess else None},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, through NVML in a background thread (a looping
    `nvidia-smi -lms` process perturbs kernel launches enough to halve the measured throughput)."""

    def __init__(self, index, period=0.02):
        self.index, self.period, self.rows, self.stop_flag, self.thread, self.ok = index, period, [], False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a list of ordinals
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except Exception:
                    phys = index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.ok = True
        except Exception:
            self.ok = False

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.rows.append((sm, mx, int(reasons)))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted({n for _, _, r in self.rows for n, bit in names.items() if r & bit})
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[1] for r in self.rows) if sm else None,
                "reasons": reasons, "samples": len(sm)}


def _event_ms(fn, reps, dev):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def measured_traffic(key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, one `ncu --set full` capture) of a kernel
    at a workload, from the committed profile summary; None when this round holds no capture for it."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        row = table["kernels"].get(key)
        if row is None:
            return None, None
        return float(row["dram_bytes_per_launch"]), f"profiles/r02_traffic.json[{key}] <- {row['from']} (commit {table.get('commit', '?')})"
    except Exception:
        return None, None


def dense_roofline(metric, Cn, d, ticks, step_ms, hbm_peak, dev, name, tick=None, grad=None):
    """Dominant kernel of c2: the FP64 dense apply (DMMA tensor path), timed alone on the engine's stream."""
    import ctypes as C
    import torch
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    a = torch.randn((Cn, d), dtype=torch.float64, device=dev)
    out = torch.empty_like(a)
    ctx = backend.context(dev)

    def gemm():
        _lib.check(lib.b2h_dense_apply(ctx, _lib.F64, backend.ptr(a), backend.ptr(metric.imm), backend.ptr(out),
                                       C.c_int64(Cn), C.c_int64(d)))
    for _ in range(3):
        gemm()
    gemm_ms = _event_ms(gemm, 20, dev)
    flops = 2.0 * Cn * d * d
    achieved = flops / (gemm_ms * 1e-3) / 1e12
    # FP64 peak is not in MEASURED_PEAKS.json: measure cuBLAS DGEMM here, the way the driver measured bf16
    n = 4096
    x = torch.randn((n, n), dtype=torch.float64, device=dev)
    y = torch.randn((n, n), dtype=torch.float64, device=dev)
    torch.matmul(x, y)
    best = min(_event_ms(lambda: torch.matmul(x, y), 1, dev) for _ in range(5))
    fp64_peak = 2.0 * n ** 3 / (best * 1e-3) / 1e12
    # the same product back to back for ~1.5 s: what the FP64 tensor path sustains under the power cap
    reps_s = max(10, int(1500.0 / best))
    fp64_sustained = 2.0 * n ** 3 / (_event_ms(lambda: torch.matmul(x, y), reps_s, dev) * 1e-3) / 1e12
    del x, y
    mm = metric.imm
    torch.matmul(a, mm)
    best = min(_event_ms(lambda: torch.matmul(a, mm), 1, dev) for _ in range(5))
    cublas_same_shape = flops / (best * 1e-3) / 1e12
    elementwise_ms = max(step_ms - ticks * 2.0 * gemm_ms, 1e-9)
    traffic, traffic_from = measured_traffic(f"dense_apply@{name}")
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
        "traffic": traffic, "traffic_from": traffic_from,
        "pipe": "FP64 tensor (DMMA.8x8x4): FP64 has no tcgen05 kind",
        "kernel": "dense_apply_dmma_async_kernel<BN> (out[C x d] = in[C x d] . M[d x d], FP64 DMMA + cp.async): "
                  "gradient and imm.g, 2 launches per tick",
        "flops_per_launch": flops, "algorithmic_bytes_per_launch": 8.0 * (2 * Cn * d + d * d), "avg_launch_ms": gemm_ms,
        "peak_source": f"measured in this run: torch.matmul fp64 {n}^3 (cuBLAS), best of 5 (MEASURED_PEAKS.json "
                       "has no FP64 figure; SURVEY.md 8d names FP64 compute as the bound of config 2)",
        "peak_sustained": fp64_sustained, "frac_of_sustained": achieved / fp64_sustained,
        "launches_per_tick": 2, "share_of_step": ticks * 2.0 * gemm_ms / step_ms,
        "cublas_same_shape_tflops": cublas_same_shape,
        # the model's gradient call (this dense apply + the potential kernel) timed inside the step, where the momentum
        # contractions of restarting chains run beside it on the side stream
        "gradient_call_in_step_ms": grad["avg_launch_us"] * 1e-3 if grad else None}
    elementwise = elementwise_roofline(tick, name, Cn, d, 8, ticks, elementwise_ms, hbm_peak)
    return roofline, elementwise


def logistic_roofline(model, Cn, d, n, ticks, step_ms, peaks, dev, dtype, name, tick=None, grad=None):
    """Dominant kernel of c3 / c5: the fused tcgen05 gradient (S product, residual, X^T R product in one kernel),
    timed through b2h_potential_and_grad on the engine's stream (includes three small side kernels)."""
    import torch
    q = torch.tensor(initial_positions("logistic", Cn, d, 12345), dtype=dtype, device=dev)
    for _ in range(3):
        model.potential_and_grad(q)
    ms_alone = _event_ms(lambda: model.potential_and_grad(q), 20 if Cn <= 8192 else 5, dev)
    # the launch time that counts is the one INSIDE the step (b2h_tick_timer around every gradient call of two engine calls):
    # a burst of a few launches runs at a higher clock than the power-capped steady state of the step
    ms = grad["avg_launch_us"] * 1e-3 if grad else ms_alone
    flops = 4.0 * n * d * Cn
    achieved = flops / (ms * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops_sustained", 1389.0))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    pieces = 2 if getattr(model, "tc_flag", 0.0) == 4.0 else 3
    traffic, traffic_from = measured_traffic(f"tc_logistic_fused16@{name}")
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_from": traffic_from,
        "kernel": ("tc_logistic_fused16_kernel" if pieces == 2 else "tc_logistic_fused_kernel") +
                  " (tcgen05.mma kind::f16 with both A operands in TMEM, TMA, one launch per tick): S = B X^T, "
                  "residual epilogue back into TMEM, G += R X",
        "flops_per_launch": flops, "avg_launch_ms": ms, "avg_launch_ms_alone": ms_alone,
        "timed": (f"inside the step: CUDA events around each of {grad['launches']} gradient calls of the engine (b2h_tick_timer)"
                  if grad else "alone, through b2h_potential_and_grad"),
        "what": f"ALGORITHMIC flops (4 N D per chain-gradient).  beta and the residual are carried as {pieces} "
                f"{'fp16' if pieces == 2 else 'bf16'} pieces for fp32-class accuracy, so the tensor pipe issues "
                f"{pieces}x these flops; timed through b2h_potential_and_grad (includes 3 small side kernels)",
        "issued_tflops": pieces * achieved, "issued_frac": pieces * achieved / peak,
        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)",
        "launches_per_tick": 1, "share_of_step": ticks * ms / step_ms}
    esize = 4 if dtype == torch.float32 else 8
    rest_ms = max(step_ms - ticks * ms, 1e-9)
    elementwise = elementwise_roofline(tick, name, Cn, d, esize, ticks, rest_ms, hbm_peak)
    return roofline, elementwise


class Dist:
    """torch.distributed plumbing of one bench process."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = dist
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        import torch
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize(self.dev)

    def reduce(self, values, op="sum"):
        import torch
        t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return t.tolist()

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def build_problem(name, dev):
    import torch
    import aehmc_b200 as ab
    kind, Cn, d, ticks, n_data = WORKLOADS[name]
    if kind == "dense":
        dtype, dtype_name = torch.float64, "f64"
        cov, prec = make_dense_problem(d)
        model = ab.models.CorrelatedGaussian(np.zeros(d), prec, device=dev)
        metric = ab.metrics.GaussianMetric(cov, dtype, dev)
    else:
        dtype, dtype_name = torch.float32, "f32"
        X, y, imm = make_logistic_problem(n_data, d)
        model = ab.models.LogisticRegression(X, y, 1.0, dtype=dtype, device=dev, tensor_core=True)
        metric = ab.metrics.GaussianMetric(imm, dtype, dev)
    return model, metric, dtype, dtype_name


def dump_rows(Cn, d, esize):
    """Chains whose [dim] rows --dump-outputs writes: all of them when the three [chains, dim] arrays fit DUMP_ROW_BYTES,
    else a fixed, seeded sample in ascending order (the same chains in every run)."""
    n = min(Cn, DUMP_ROW_BYTES // (3 * d * esize))
    if n == Cn:
        return np.arange(Cn)
    return np.sort(np.random.default_rng(0).choice(Cn, n, replace=False))


def _host_float(t):
    a = t.detach().cpu().numpy()
    return a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)     # int / bool: exact in float64


def last_step_outputs(info, extras, rows, chain_offset=0):
    """Host copies of what one engine call returned to its caller: the [chains, dim] arrays at `rows` only, every
    per-chain array in full, the call's counters (leapfrogs, transitions, ticks, chain-ticks) and the global ids of
    `rows` as `chains`.  Float arrays keep their dtype; integer and boolean arrays become float64."""
    import torch
    st = info.state
    idx = torch.from_numpy(np.asarray(rows, dtype=np.int64)).to(st.position.device)
    out = {"chains": (chain_offset + np.asarray(rows)).astype(np.float64)}
    for k in ("position", "momentum", "potential_energy_grad"):
        out[k] = _host_float(getattr(st, k).index_select(0, idx))
    out["potential_energy"] = _host_float(st.potential_energy)
    for k in ("acceptance_probability", "num_doublings", "is_turning", "is_diverging"):
        out[k] = _host_float(getattr(info, k))
    out["n_leapfrog"] = _host_float(extras["n_leapfrog"])
    out["counters"] = _host_float(extras["counters"])
    return out


def write_outputs(path, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"outputs of {total} bytes exceed the {DUMP_BYTES}-byte limit of --dump-outputs")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def run_tick_workload(name, D, steps, warmup, min_timed_s=0.0, with_e2e=True, dump=False):
    """Device-resident and end-to-end throughput of one tick-engine workload.  Returns a dict (rank-reduced)."""
    import torch
    import aehmc_b200 as ab
    from aehmc_b200 import _engine

    kind, Cn, d, ticks, n_data = WORKLOADS[name]
    eps = EPS[kind]
    dev = D.dev
    model, metric, dtype, dtype_name = build_problem(name, dev)
    chain_offset = D.rank * Cn
    q_host = torch.from_numpy(initial_positions(kind, Cn, d, chain_offset)).to(dtype).pin_memory()
    srng = ab.RandomStream(seed=2026, chain_offset=chain_offset)
    key = ("bench", name, D.rank)
    esize = q_host.element_size()

    # ---- device-resident arm: state lives in the engine workspace, each step continues it -----------------
    state = ab.nuts.new_state(q_host.to(dev), model)
    info, extras = _engine.run("nuts", model, metric, srng, state, eps, max_ticks=ticks, workspace_key=key,
                               return_counters=True)
    state = info.state
    last = {}

    def step_resident():
        nonlocal state
        info, ex = _engine.run("nuts", model, metric, srng, state, eps, max_ticks=ticks, resume=True,
                               workspace_key=key, return_counters=True)
        state = info.state
        last["info"], last["extras"] = info, ex
        return ex["counters"]

    warm = max(warmup, 3)
    for _ in range(warm):
        step_resident()
    if min_timed_s > 0:                     # secondary workloads: enough steps for a timed region of min_timed_s
        est = _event_ms(step_resident, 3, dev)
        steps = int(min(max(steps, math.ceil(min_timed_s * 1e3 / max(est, 1e-3))), 2000))
    D.barrier()
    sampler = ClockSampler(D.local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    ev0.record()
    counters = []
    for _ in range(steps):
        counters.append(step_resident())
    ev1.record()
    D.barrier()
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    # every engine call returns fresh tensors: these are the last timed call's, copied out before the extra calls below
    outputs = last_step_outputs(last["info"], last["extras"], dump_rows(Cn, d, esize), chain_offset) if dump else None
    cnt = torch.stack(counters).sum(0).cpu().numpy()      # leapfrogs, transitions, ticks(unused), chain-ticks
    acc = last["info"].acceptance_probability
    ms_total = D.reduce([ms_total], "max")[0]
    total_leapfrogs, total_transitions, acc_sum = D.reduce([cnt[0], cnt[1], float(acc.sum())])
    value = total_leapfrogs / (ms_total * 1e-3)
    out = {"name": name, "kind": kind, "chains_per_gpu": Cn, "dim": d, "n_data": n_data, "ticks": ticks, "eps": eps,
           "steps": steps, "warmup": warm, "value": value, "ms_per_step": ms_total / steps, "ms_total": ms_total,
           "dtype": dtype, "dtype_name": dtype_name, "clocks": clocks, "model": model, "metric": metric,
           "transitions_per_step": total_transitions / steps,
           "mean_leapfrogs_per_transition": total_leapfrogs / max(total_transitions, 1.0),
           "mean_accept": acc_sum / (Cn * D.world), "esize": esize, "q_host": q_host, "chain_offset": chain_offset,
           "outputs": outputs}

    # ---- the tick kernel (integrator + U-turn + proposal bookkeeping of one leapfrog of every chain) timed on its own:
    #      b2h_tick_timer brackets each of its launches with CUDA events on the engine's stream (outside the headline
    #      region above: the events would serialise nothing, but they are not part of the product path)
    out["tick_kernel"] = time_tick_kernel(step_resident, dev)
    out["gradient_in_step"] = time_tick_kernel(step_resident, dev, what=2)

    # ---- end-to-end arm: host buffers in, host buffers out, through the public API ----------------------
    if with_e2e:
        q_out = torch.empty((Cn, d), dtype=dtype).pin_memory()
        acc_out = torch.empty(Cn, dtype=torch.float64).pin_memory()

        def step_e2e():
            q_dev = q_host.to(dev, non_blocking=True)
            st = ab.nuts.new_state(q_dev, model)
            info, ex = _engine.run("nuts", model, metric, srng, st, eps, max_ticks=ticks, workspace_key=key,
                                   return_counters=True)
            q_out.copy_(info.state.position, non_blocking=True)
            acc_out.copy_(info.acceptance_probability, non_blocking=True)
            return ex["counters"]

        for _ in range(3):
            step_e2e()
        D.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        cs = [step_e2e() for _ in range(steps)]
        e1.record()
        D.barrier()
        ms_e2e = D.reduce([e0.elapsed_time(e1)], "max")[0]
        leap_e2e = D.reduce([float(torch.stack(cs).sum(0)[0].item())])[0]
        out["e2e"] = {"value": leap_e2e / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(Cn * d * esize),
                      "d2h_bytes_per_step": int(Cn * d * esize + Cn * 8), "seconds": ms_e2e * 1e-3,
                      "what": "pinned host positions -> device, new_state, TICKS ticks, position + acceptance back to "
                              "pinned host"}
    _engine.release_workspace(key)
    return out


def time_tick_kernel(step, dev, steps=2, what=1):
    """Average duration of the split engine's tick kernel (what = 1) or of its gradient call (what = 2: the model's
    contraction kernels with their side kernels) over `steps` engine calls: CUDA events around every launch, in the step."""
    import ctypes as C
    from aehmc_b200 import _lib, backend
    lib = _lib.load()
    ctx = backend.context(dev)
    _lib.check(lib.b2h_tick_timer(ctx, what))
    for _ in range(steps):
        step()
    ms, n = C.c_double(0.0), C.c_int64(0)
    _lib.check(lib.b2h_tick_timer_read(ctx, C.byref(ms), C.byref(n)))
    _lib.check(lib.b2h_tick_timer(ctx, 0))
    if n.value == 0:
        return None
    return {"avg_launch_us": ms.value * 1e3 / n.value, "launches": int(n.value)}


def elementwise_roofline(tick, name, Cn, d, esize, ticks, rest_ms, hbm_peak):
    """HBM roofline of the tick kernel.  `achieved` = ALGORITHMIC bytes (SURVEY.md 8d: 11*d*s per chain-tick, NUTS
    inner step with U-turn bookkeeping) over the kernel's measured launch time; `traffic` = the DRAM bytes one launch
    really moves (ncu), with the bandwidth that corresponds to it."""
    alg = 11.0 * d * esize * Cn
    tr = measured_traffic(f"tile_tick@{name}")
    if tick is not None:
        sec = tick["avg_launch_us"] * 1e-6
        how = (f"11*d*{esize} algorithmic bytes per chain-tick x {Cn} chains over the tick kernel's average launch time, "
               f"CUDA events around each of {tick['launches']} launches (b2h_tick_timer)")
    else:                                   # register-front kernels (B2H_TILE_TICK=0) or no split engine: by subtraction
        sec = rest_ms * 1e-3 / ticks
        how = f"derived: 11*d*{esize} algorithmic bytes per chain-tick over (step time - contraction time) / ticks"
    achieved = alg / sec / 1e9
    row = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
           "traffic": tr[0], "traffic_from": tr[1], "how": how,
           "kernel": "tile_tick_kernel (engine_tile.inl): kick, kinetic energy, momentum sums, U-turn checkpoints and dot "
                     "products, progressive / biased sampling, sub-tree and transition ends, half kick + drift of the "
                     "next leapfrog -- one launch per tick",
           "algorithmic_bytes_per_launch": alg, "avg_launch_us": sec * 1e6,
           "everything_but_contractions_ms_per_tick": rest_ms / ticks}
    if tr[0] is not None:
        row["traffic_gbs"] = tr[0] / sec / 1e9
        row["traffic_frac"] = tr[0] / sec / 1e9 / hbm_peak
    return row


def rooflines_for(w, D, peaks):
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    if w["kind"] == "dense":
        return dense_roofline(w["metric"], w["chains_per_gpu"], w["dim"], w["ticks"], w["ms_per_step"], hbm_peak, D.dev,
                              w["name"], w.get("tick_kernel"), w.get("gradient_in_step"))
    return logistic_roofline(w["model"], w["chains_per_gpu"], w["dim"], w["n_data"], w["ticks"], w["ms_per_step"], peaks,
                             D.dev, w["dtype"], w["name"], w.get("tick_kernel"), w.get("gradient_in_step"))


def ess_leg(w, D, args):
    """Second BASELINE metric (NUTS ESS/s) and the diagnostics exchange of configs[4], all inside timed regions:
    pooled warm-up (adaptation statistics merged over the ranks) -> KEEP stored transitions -> rank-normalised split
    bulk-ESS and R-hat (arviz defaults) of the monitored coordinates over all chains of all ranks."""
    import torch
    import aehmc_b200 as ab
    from aehmc_b200 import _engine
    dev, model, Cn, d = D.dev, w["model"], w["chains_per_gpu"], w["dim"]
    keep, warm = args.ess_transitions, args.ess_warmup
    kernel = ab.nuts.new_kernel(ab.RandomStream(seed=7, chain_offset=w["chain_offset"]), model)
    st0 = ab.nuts.new_state(w["q_host"].to(dev), model)
    imm0 = w["metric"].imm if w["kind"] == "logistic" else None
    full = w["kind"] == "dense"

    def timed(fn):
        D.barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        r = fn()
        s1.record()
        D.barrier()
        return r, D.reduce([s0.elapsed_time(s1)], "max")[0] * 1e-3

    (state, (eps, imm), winfo), t_warm = timed(lambda: ab.window_adaptation.run(
        kernel, st0, warm, pooled=True, is_mass_matrix_full=full, initial_inverse_mass_matrix=imm0,
        initial_step_size=w["eps"]))
    # one step size for all chains (the median of the per-chain dual-averaging results): with per-chain step sizes the
    # chains with the smallest ones build the deepest trees and the whole batch waits for them
    eps = torch.full_like(eps, float(eps.median()))
    (info, ex), t_sample = timed(lambda: _engine.run("nuts", model, imm, kernel.spec["srng"], state, eps,
                                                      n_transitions=keep, store_draws=keep, return_counters=True))
    dims = list(range(min(8, d)))
    draws = ex["draws"]

    def diagnostics():
        return ab.diagnostics.ess(draws, dims=dims), ab.diagnostics.rhat(draws, dims=dims)
    (ess, rhat), t_diag = timed(diagnostics)
    leap = D.reduce([float(ex["counters"][0].item())])[0]
    acc = D.reduce([float(info.acceptance_probability.sum())])[0] / (Cn * D.world)
    eps_med = float(eps.median())
    del draws, ex
    torch.cuda.empty_cache()
    ess_min, rhat_max = float(np.nanmin(ess)), float(np.nanmax(rhat))
    return {
        "nuts_ess_per_sec": ess_min / t_sample, "rhat_max": rhat_max, "ess_min": ess_min,
        "ess_how": f"pooled window adaptation ({warm} transitions, initial inverse mass matrix "
                   f"{'4/N' if imm0 is not None else 'identity'}, statistics merged over the ranks) then {keep} kept NUTS "
                   "transitions per chain at the median adapted step size; rank-normalised split bulk-ESS and R-hat (arviz defaults) of the first "
                   f"{len(dims)} coordinates over all chains of all ranks, minimum ESS divided by the sampling time of the "
                   "kept transitions",
        "warmup_seconds": t_warm, "sampling_seconds": t_sample, "diagnostics_seconds": t_diag,
        "mean_accept_after_warmup": acc, "step_size_median_after_warmup": eps_med,
        "pooled_window_sizes": winfo.get("pooled_window_sizes"),
        "e2e_with_diagnostics": {
            "value": leap / (t_sample + t_diag), "unit": UNIT, "seconds": t_sample + t_diag,
            "what": f"{keep} stored NUTS transitions of every chain + the diagnostics exchange (per-rank sort, all-gather "
                    "of the sorted monitored draws for the global rank normalisation, all-reduce of the autocovariance "
                    "sufficient statistics) + host ESS / R-hat arithmetic, timed together, max over ranks",
            "collectives": "nccl all_gather + all_reduce" if D.world > 1 else "none at N = 1 (same code path)"}}


def secondary_c4(D, peaks):
    """configs[3]: window_adaptation (1000 steps) + 1000 NUTS draws, 10-dim funnel and eight schools, 65536 chains."""
    import torch
    import aehmc_b200 as ab
    from aehmc_b200 import _engine, metrics
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    Cn, W, Dn = 65536, 1000, 1000
    out = {}
    for name, model in (("funnel", ab.models.NealFunnel(10, device=D.dev)), ("eight_schools", ab.models.EightSchools(device=D.dev))):
        q0 = np.random.default_rng(0).standard_normal((Cn, 10))
        kernel = ab.nuts.new_kernel(ab.RandomStream(seed=11), model)
        state = ab.nuts.new_state(q0, model)
        res = {}

        def warm():
            res["w"] = ab.window_adaptation.run(kernel, state, W)
        ms_w = _event_ms(warm, 1, D.dev)
        wstate, (eps, imm), _ = res["w"]

        def draw():
            res["d"] = _engine.run("nuts", model, metrics.per_chain(imm), kernel.spec["srng"], wstate, eps,
                                   n_transitions=Dn, store_draws=Dn, return_counters=True)
        # the 7 GB of draw / statistics storage come from torch's caching allocator: take them from the driver once,
        # outside the timed call (a cudaMalloc of that size costs 0.1-0.2 s of host time, a third of the eight-schools run)
        pre = [torch.empty((Dn, Cn, 10), dtype=torch.float64, device=D.dev), torch.empty((Dn, Cn, 4), dtype=torch.float64, device=D.dev)]
        del pre
        ms_d = _event_ms(draw, 1, D.dev)
        info, ex = res["d"]
        leap = int(ex["counters"][0].item())
        per_chain = ex["draw_stats"][:, :, 2].sum(0)
        tail = {"mean": float(per_chain.mean()), "p99": float(torch.quantile(per_chain, 0.99)),
                "max": float(per_chain.max())}
        ex = None
        res["d"] = (info, None)
        torch.cuda.empty_cache()
        # the same chains free-running for the mean number of leapfrogs: every lane busy all the time (throughput of the
        # kernel), against the fixed-number-of-transitions run above, which ends with its slowest chains
        ticks = max(int(tail["mean"]), 1)

        def free():
            res["f"] = _engine.run("nuts", model, metrics.per_chain(imm), kernel.spec["srng"], wstate, eps,
                                   max_ticks=ticks, return_counters=True)
        ms_f = _event_ms(free, 1, D.dev)
        leap_f = int(res["f"][1]["counters"][0].item())
        out[name] = {"value": leap / (ms_d * 1e-3), "unit": UNIT, "chains": Cn, "warmup_ms": ms_w, "sampling_ms": ms_d,
                     "sampling_leapfrogs": leap, "transitions_per_sec": Cn * Dn / (ms_d * 1e-3),
                     "per_chain_leapfrogs": tail,
                     "free_running": {"value": leap_f / (ms_f * 1e-3), "unit": UNIT, "ticks": ticks, "ms": ms_f,
                                      "what": "every chain takes `ticks` leapfrogs (transitions restart independently): "
                                              "the kernel's throughput without the tail of the slowest chains"},
                     "roofline": {"bound": "hbm", "achieved": leap * 11 * 10 * 8 / (ms_d * 1e-3) / 1e9, "peak": hbm_peak,
                                  "unit": "GB/s", "frac": leap * 11 * 10 * 8 / (ms_d * 1e-3) / 1e9 / hbm_peak,
                                  "frac_free_running": leap_f * 11 * 10 * 8 / (ms_f * 1e-3) / 1e9 / hbm_peak,
                                  "what": "11*d*s algorithmic bytes per leapfrog (SURVEY 8d); the state of a chain "
                                          "stays on chip in the persistent kernel (latency / divergence bound, SURVEY 8d), "
                                          "HBM sees only draws out"},
                     "step_size_median": float(eps.median()),
                     "mean_accept": float(info.acceptance_probability.mean()),
                     "last_transition_depth_hist": torch.bincount(info.num_doublings.long(), minlength=11).cpu().tolist(),
                     "last_transition_divergent_frac": float(info.is_diverging.double().mean())}
        del res
    return {"workload": f"c4 (BASELINE.json configs[3]): window_adaptation({W}) + {Dn} NUTS draws, d = 10, {Cn} chains, "
                        "f64, persistent fused kernel", **out}


def secondary_c1(D, peaks):
    """configs[0]: HMC, velocity_verlet, L = 10, diagonal imm, 100-dim iid Gaussian: 1 chain (the reference's own
    configuration) and 65536 chains, next to the single-threaded CPU oracle."""
    import aehmc_b200 as ab
    from aehmc_b200 import _engine
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    d, sigma = make_c1_problem()
    L = 10
    model = ab.models.IIDGaussian(np.zeros(d), sigma, device=D.dev)
    out = {"workload": "c1 (BASELINE.json configs[0]): HMC velocity_verlet L=10, d=100 iid Gaussian, diagonal imm, f64"}
    for Cn, n_tr in ((1, 1000), (65536, 400)):
        q0 = np.random.default_rng(2).standard_normal((Cn, d))
        srng = ab.RandomStream(seed=1)
        state = ab.hmc.new_state(q0, model)
        res = {}

        def run():
            res["r"] = _engine.run("hmc", model, sigma ** 2, srng, state, 0.25, n_transitions=n_tr,
                                   num_integration_steps=L, store_draws=n_tr if Cn == 1 else 0)
        run()
        # three timed calls, the fastest reported (all three kept): a single call right after the c4 leg was seen at
        # 220 - 360 ms against 149 - 165 ms for the same work (benchmarks/c1_only.py)
        ms_all = [_event_ms(run, 1, D.dev) for _ in range(3)]
        ms = min(ms_all)
        info, ex = res["r"]
        evals = Cn * n_tr * L
        row = {"value": evals / (ms * 1e-3), "unit": UNIT, "transitions": n_tr, "ms": ms, "ms_all": ms_all,
               "mean_accept": float(info.acceptance_probability.mean()),
               "roofline": {"bound": "hbm", "achieved": evals * 6 * d * 8 / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": evals * 6 * d * 8 / (ms * 1e-3) / 1e9 / hbm_peak,
                            "what": "6*d*s algorithmic bytes per leapfrog (SURVEY 8d); the trajectory stays in registers"}}
        if Cn == 1:
            ess = host_ess(ex["draws"].double().cpu().numpy()[:, :, :8])
            row["ess_per_sec"] = None if ess is None else ess / (ms * 1e-3)
        out[f"chains_{Cn}"] = row
    out["cpu_baseline"] = cpu_c1_sample()
    return out


def secondary_tick(name, D, args, peaks):
    import torch
    w = run_tick_workload(name, D, args.steps, args.warmup, min_timed_s=MIN_TIMED_S, with_e2e=True)
    roofline, elementwise = rooflines_for(w, D, peaks)
    out = {"workload": describe(name), "value": w["value"], "unit": UNIT, "ms_per_step": w["ms_per_step"],
           "steps": w["steps"], "timed_seconds": w["ms_total"] * 1e-3, "ticks_per_step": w["ticks"], "dtype": w["dtype_name"],
           "mean_accept": w["mean_accept"], "mean_leapfrogs_per_transition": w["mean_leapfrogs_per_transition"],
           "e2e": w["e2e"], "clocks": w["clocks"], "roofline": roofline, "roofline_elementwise": elementwise}
    del w
    torch.cuda.empty_cache()
    return out


def run_gpu_arm(args):
    import torch
    D = Dist()
    peaks = load_peaks()
    name = args.workload
    w = run_tick_workload(name, D, args.steps, args.warmup, dump=args.dump_outputs is not None)
    if args.dump_outputs is not None and D.rank == 0:
        write_outputs(args.dump_outputs, w.pop("outputs"))
    roofline, roofline_elementwise = rooflines_for(w, D, peaks)
    kind, Cn, d, ticks = w["kind"], w["chains_per_gpu"], w["dim"], w["ticks"]
    kernels_per_tick = 6 if kind == "dense" else 4
    # dense: tick kernel, gradient apply, potential, imm.g apply, momentum rider GEMM + its reduce
    # logistic: tick kernel, beta split, fused gradient, finish (profiles/r02_launches_c5.md)

    ess = {}
    if not args.no_ess:
        ess = ess_leg(w, D, args)

    secondary = None
    if D.world == 1 and not args.no_secondary:
        model = w.pop("model"); metric = w.pop("metric")
        del model, metric
        torch.cuda.empty_cache()
        secondary = {}
        for sec in [s for s in ("c3", "c2") if s != name]:
            try:
                secondary[sec] = secondary_tick(sec, D, args, peaks)
            except Exception as e:                                   # a secondary failure must not lose the headline
                secondary[sec] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
        for sec, fn in (("c4", secondary_c4), ("c1", secondary_c1)):
            try:
                secondary[sec] = fn(D, peaks)
            except Exception as e:
                secondary[sec] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()

    if D.rank == 0:
        line = {
            "metric": METRIC, "value": w["value"], "unit": UNIT, "n_gpus": D.world, "steps": w["steps"],
            "warmup": w["warmup"], "ms_per_step": w["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": w["dtype_name"], "data": "synthetic",
            "config": {"workload": describe(name), "chains_per_gpu": Cn, "chains_total": Cn * D.world, "dim": d,
                       "step_size": w["eps"], "max_num_expansions": 10, "ticks_per_step": ticks, "rng": "philox4x32-10",
                       "l2": "engine state larger than the 126 MB L2 (no flush needed)" if kind == "dense" else
                             "the design matrix X (25.6 MB fp16) is meant to stay L2-resident; the chain state "
                             f"({Cn} x {d} x ~20 arrays) " + ("exceeds L2" if Cn * d * 80 > 126e6 else "fits L2"),
                       "timed_seconds": w["ms_total"] * 1e-3,
                       "mean_accept": w["mean_accept"],
                       "transitions_per_step": w["transitions_per_step"],
                       "mean_leapfrogs_per_transition": w["mean_leapfrogs_per_transition"]},
            "e2e": w["e2e"],
            "gpu_launches": int(w["steps"] * (ticks * kernels_per_tick + 3)),
            "clocks": w["clocks"],
            "roofline": roofline, "roofline_elementwise": roofline_elementwise,
        }
        line.update(ess)
        if secondary is not None:
            line["secondary"] = secondary
        if D.world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            n_tr = cpu_transitions(name)
            r = cpu_reference_sample(name, cores, n_tr)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "port",
                                    "ess_per_sec": r["ess_per_sec"], "mean_accept": r["mean_accept"],
                                    "sample": f"{cores} oracle chains (one per core) x {n_tr} NUTS transitions, "
                                              f"{r['leapfrogs']} leapfrogs in {r['wall_s']:.1f} s wall"}
        print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-ess", action="store_true", help="skip the ESS/s + diagnostics leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads (c3, c2, c4, c1)")
    ap.add_argument("--ess-transitions", type=int, default=200, help="kept NUTS transitions of the ESS leg")
    ap.add_argument("--ess-warmup", type=int, default=100, help="pooled window-adaptation transitions before them")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0's chains; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
