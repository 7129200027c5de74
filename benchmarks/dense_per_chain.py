"""Per-chain dense inverse mass matrices: the batched per-chain mat-vec, NUTS with one dense metric per chain against a
per-chain diagonal and one pooled dense metric, and the per-chain dense warm-up.

    python benchmarks/dense_per_chain.py [--out FILE] [--quick]

 - mat-vec: b2h_dense_apply_per_chain (tri = 0) at (C, d) = (4096, 128), (65536, 32), (131072, 16), (4096, 64), FP64
   and FP32; kernel time from CUDA events over a window of at least 1 s.  Bytes = C d^2 s (the matrices; the input
   and output rows add 2 C d s), reported as GB/s and as a fraction of the 7.7 TB/s HBM data-sheet peak.  Rows whose
   matrices fit the 126 MB L2 are flagged: they are served from L2 after the first launch.
 - NUTS: correlated Gaussian, d = 32, covariance eigenvalues log-spaced over [1e-3, 1] in a random orientation
   (condition number 1e3), 4096 and 65536 chains, FP64.  Each metric is adapted by window adaptation (1000 steps:
   per-chain dense, per-chain diagonal, pooled dense), then 100 transitions are sampled: gradient evaluations per
   second (leapfrogs of all chains over wall time) and bulk ESS (minimum over the dimensions) per gradient evaluation.
 - warm-up: wall time of 1000 per-chain dense warm-up steps at 4096 chains, d = 32.
Prints one JSON object per line; the GPU name and power limit come first."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import aehmc_b200 as ab  # noqa: E402
from aehmc_b200 import _lib, backend  # noqa: E402

HBM_PEAK_GBS = 7700.0        # HGX B200 data sheet, one GPU
L2_BYTES = 126e6


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def timed(fn, min_s=1.0):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    reps = max(10, int(math.ceil(min_s / max(e0.elapsed_time(e1) * 1e-3, 1e-6))))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def matvec_rows(quick):
    lib = _lib.load()
    shapes = [(4096, 128), (65536, 32), (131072, 16), (4096, 64)]
    for Cn, d in shapes[:1] if quick else shapes:
        for dt in (torch.float64, torch.float32):
            x = torch.randn(Cn, d, dtype=dt, device="cuda")
            M = torch.randn(Cn, d, d, dtype=dt, device="cuda")
            out = torch.empty_like(x)
            ctx = backend.context(x.device)

            def call():
                _lib.check(lib.b2h_dense_apply_per_chain(ctx, backend.code(dt), backend.ptr(x), backend.ptr(M),
                                                         backend.ptr(out), C.c_int64(Cn), C.c_int64(d), C.c_int32(0)))
            ms = timed(call)
            ref = torch.einsum("ck,ckj->cj", x.double(), M.double())
            err = float((out.double() - ref).abs().max() / ref.abs().max())
            mbytes = Cn * d * d * x.element_size()
            gbs = mbytes / (ms * 1e-3) / 1e9
            yield {"bench": "matvec", "C": Cn, "d": d, "dtype": str(dt).split(".")[1], "ms": round(ms, 4),
                   "matrix_bytes": mbytes, "GB_per_s": round(gbs, 1), "frac_hbm_peak": round(gbs / HBM_PEAK_GBS, 3),
                   "l2_resident": mbytes < L2_BYTES, "max_rel_err_vs_fp64": err}
            del x, M, out, ref
            torch.cuda.empty_cache()


def _target(d, seed=0):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((d, d)))
    cov = (Q * np.logspace(0, -3, d)) @ Q.T
    cov = 0.5 * (cov + cov.T)
    return cov, ab.models.CorrelatedGaussian(np.zeros(d), np.linalg.inv(cov))


def nuts_rows(quick):
    d, warm, n = 32, (200 if quick else 1000), 100
    cov, model = _target(d)
    for Cn in (4096,) if quick else (4096, 65536):
        q0 = np.random.default_rng(1).standard_normal((Cn, d)) * 0.1
        for which in ("per_chain_dense", "per_chain_diag", "pooled_dense"):
            kernel = ab.nuts.new_kernel(ab.RandomStream(seed=2), model)
            full, pooled = which != "per_chain_diag", which == "pooled_dense"
            state, (eps, imm), _ = ab.window_adaptation.run(kernel, ab.nuts.new_state(q0, model), warm,
                                                            is_mass_matrix_full=full, pooled=pooled)
            metric = imm if pooled else ab.metrics.per_chain(imm)
            ab.sampling.sample(kernel, state, eps, metric, 2, store_draws=False)        # warm the shapes
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            info, draws, stats, _ = ab.sampling.sample(kernel, state, eps, metric, n)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            grads = float(stats[:, :, 2].sum())
            ess = ab.diagnostics.ess(draws, distributed=False)
            ess_min = float(torch.as_tensor(ess).min())
            yield {"bench": "nuts", "metric": which, "C": Cn, "d": d, "cond": 1e3, "warmup_steps": warm,
                   "transitions": n, "wall_s": round(wall, 3), "grad_evals_per_s": round(grads / wall, 1),
                   "mean_leapfrogs": round(grads / (n * Cn), 2), "ess_min": round(ess_min, 1),
                   "ess_per_grad_eval": ess_min / grads, "median_step_size": float(eps.median())}
            del state, imm, draws, stats
            torch.cuda.empty_cache()


def warmup_rows(quick):
    d, Cn, steps = 32, 4096, (200 if quick else 1000)
    cov, model = _target(d)
    q0 = np.random.default_rng(3).standard_normal((Cn, d)) * 0.1
    kernel = ab.nuts.new_kernel(ab.RandomStream(seed=4), model)
    ab.window_adaptation.run(kernel, ab.nuts.new_state(q0[:64], model), 30, is_mass_matrix_full=True)   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    state, (eps, imm), _ = ab.window_adaptation.run(kernel, ab.nuts.new_state(q0, model), steps,
                                                    is_mass_matrix_full=True)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    err = np.linalg.norm(imm.cpu().numpy() - cov, axis=(1, 2)) / np.linalg.norm(cov)
    yield {"bench": "warmup", "metric": "per_chain_dense", "C": Cn, "d": d, "steps": steps, "wall_s": round(wall, 3),
           "median_rel_frobenius_err": float(np.median(err))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_dense_per_chain.jsonl"))
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for row in [gpu_info()]:
            print(json.dumps(row), flush=True); f.write(json.dumps(row) + "\n")
        for gen in (matvec_rows, nuts_rows, warmup_rows):
            for row in gen(a.quick):
                print(json.dumps(row), flush=True); f.write(json.dumps(row) + "\n"); f.flush()


if __name__ == "__main__":
    main()
