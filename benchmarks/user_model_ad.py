"""Automatic differentiation of user log-densities: forward mode (dual numbers) against reverse mode (per-chain tape).

    python benchmarks/user_model_ad.py [--out FILE] [--quick]

Densities: the test suite's funnel and its data-carrying logistic regression (tests/test_gpu_user_model.py).
 - d in {16, 32, 64}: forward against reverse (reverse reached below its dim-64 boundary through the C-ABI);
 - d in {128, 256, 1000}: reverse only;
 each at 4096 and 65536 chains, FP64.  Per row: ms per gradient of all chains (CUDA events over a window of at least
 1 s), tape nodes per chain, the tape traffic per gradient computed from the node count and the layout, and that
 traffic over the time against the HBM peak bench.py uses.
 - NUTS gradient evaluations per second on the funnel at d = 1000 with 4096 chains, reverse mode against the
 built-in NealFunnel.
Prints one JSON object per line; the GPU name and power limit come first."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import aehmc_b200 as ab  # noqa: E402
from aehmc_b200 import _engine, _lib, backend  # noqa: E402
from test_gpu_user_model import FUNNEL_DENSITY, LOGISTIC_DENSITY  # noqa: E402

N_DATA = 16                  # logistic rows: each adds ~2d tape nodes per chain
TAPE_BYTES_CAP = 40e9        # rows whose tape would exceed this are reported, not run


class ReverseUserModel(ab.models.UserModel):
    FORWARD_MAX_DIM = 0


def hbm_peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
    except Exception:
        return 6650.0


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def tape_traffic(nodes, d, Cn, es):
    """Bytes the tape moves in one gradient of Cn chains: every node is written once while recording (two int32 ids,
    two partials, its zeroed adjoint) and read once in the sweep (ids, partials, adjoint) with two adjoint
    read-modify-writes; the input adjoints are zeroed and read once."""
    return Cn * (nodes * ((8 + 3 * es) + (8 + 3 * es) + 4 * es) + d * 2 * es)


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
    return e0.elapsed_time(e1) / reps, reps


def gradient_row(model, mode, density, d, Cn):
    lib = _lib.load()
    q = torch.tensor(0.5 * np.random.default_rng(d).standard_normal((Cn, d)), dtype=model.dtype, device="cuda")
    U = torch.empty(Cn, dtype=model.dtype, device="cuda")
    g = torch.empty_like(q)
    m = model.struct()
    code = backend.code(model.dtype)
    nbytes = lib.b2h_potential_workspace_bytes(C.byref(m), code, C.c_int64(Cn))
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device="cuda")
    ctx = backend.context(model.device)

    def call():
        _lib.check(lib.b2h_potential_and_grad(ctx, C.byref(m), code, backend.ptr(q), backend.ptr(U), backend.ptr(g),
                                              C.c_int64(Cn), backend.ptr(ws), C.c_int64(ws.numel())))
    ms, reps = timed(call)
    model.check_tape()
    row = {"density": density, "mode": mode, "d": d, "chains": Cn, "ms_per_gradient": ms, "reps": reps,
           "window_s": ms * reps * 1e-3, "workspace_bytes": int(nbytes)}
    if mode == "reverse":
        es = q.element_size()
        tb = tape_traffic(model.tape_nodes, d, Cn, es)
        row.update(tape_nodes_per_chain=model.tape_nodes, tape_bytes_per_gradient=tb, tape_gbs=tb / (ms * 1e-3) / 1e9,
                   tape_frac_of_hbm_peak=tb / (ms * 1e-3) / 1e9 / hbm_peak_gbs())
    return row


def logistic_data(d):
    rng = np.random.default_rng(100 + d)
    X = rng.standard_normal((N_DATA, d)) / np.sqrt(d)
    y = (rng.random(N_DATA) < 0.5).astype(np.float64)
    return np.concatenate([[N_DATA], X.ravel(), y])


def nuts_rate(model, d, Cn, transitions):
    q0 = 0.5 * np.random.default_rng(7).standard_normal((Cn, d))
    state = ab.nuts.new_state(q0, model)
    srng = ab.RandomStream(seed=3)
    key = ("bench", id(model))
    _engine.run("nuts", model, np.ones(d), srng, state, 0.1, n_transitions=1, workspace_key=key)   # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    info, extras = _engine.run("nuts", model, np.ones(d), srng, state, 0.1, n_transitions=transitions,
                               workspace_key=key, return_counters=True)
    e1.record()
    torch.cuda.synchronize()
    _engine.release_workspace(key)
    s = e0.elapsed_time(e1) * 1e-3
    evals = int(extras["counters"][0].item())
    return {"chains": Cn, "d": d, "transitions": transitions, "seconds": s, "gradient_evals": evals,
            "evals_per_s": evals / s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--quick", action="store_true", help="one chain count, small dims (a dry run)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    out = open(a.out, "a") if a.out else None

    def emit(obj):
        line = json.dumps(obj)
        print(line, flush=True)
        if out:
            out.write(line + "\n"); out.flush()

    emit(dict(gpu_info(), hbm_peak_gbs=hbm_peak_gbs(), dtype="float64"))
    chains = (4096,) if a.quick else (4096, 65536)
    for density, src in (("funnel", FUNNEL_DENSITY), ("logistic", LOGISTIC_DENSITY)):
        for d in ((16, 128) if a.quick else (16, 32, 64, 128, 256, 1000)):
            data = logistic_data(d) if density == "logistic" else None
            modes = ("forward", "reverse") if d <= 64 else ("reverse",)
            for mode in modes:
                cls = ab.models.UserModel if mode == "forward" else ReverseUserModel
                model = cls(src, d, data=data, autodiff=True)
                for Cn in chains:
                    if mode == "reverse":
                        tb = model.tape_nodes * ((Cn + 31) // 32 * 32) * 32
                        if tb > TAPE_BYTES_CAP:
                            emit({"density": density, "mode": mode, "d": d, "chains": Cn, "skipped":
                                  f"tape of {tb / 1e9:.0f} GB", "tape_nodes_per_chain": model.tape_nodes})
                            continue
                    emit(gradient_row(model, mode, density, d, Cn))
                del model
                torch.cuda.empty_cache()
    d, Cn = (128, 512) if a.quick else (1000, 4096)
    for name, model in (("funnel reverse-mode UserModel", ab.models.UserModel(FUNNEL_DENSITY, d, autodiff=True)),
                        ("built-in NealFunnel", ab.models.NealFunnel(d))):
        emit(dict(nuts_rate(model, d, Cn, 1 if a.quick else 3), model=name))


if __name__ == "__main__":
    main()
