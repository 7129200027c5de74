"""Warp-per-chain user log-densities against thread-per-chain ones.

    python benchmarks/user_model_warp.py [--out FILE] [--quick]

Densities (tests/warp_sources.py, tests/test_gpu_user_model.py): the funnel and the data-carrying logistic regression,
each in the thread form and the warp form with reverse-mode autodiff, and a hand-written funnel in both forms.
 - Gradient timings: d in {128, 1000, 4096} x chains in {4096, 65536}, ms per gradient of all chains (CUDA events over
   a window of at least 1 s), FP64.  Reverse rows give the tape nodes per chain (thread) or per lane (warp), the tape
   traffic per gradient computed from the node count and the layout, and that traffic over the time against the HBM
   peak; hand-written rows give 2 d s C bytes (q read, g written) over the time.  Rows whose tape would exceed
   TAPE_BYTES_CAP are reported, not run.
 - NUTS gradient evaluations per second on the funnel at d = 1000 with 4096 chains: thread reverse, warp reverse, warp
   hand-written and the built-in NealFunnel.
Prints one JSON object per line; the GPU name and power limit come first."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
import user_model_ad as r03  # noqa: E402  (puts the repository and tests/ on the path)
from aehmc_b200 import _lib, backend  # noqa: E402
from test_gpu_user_model import FUNNEL_DENSITY, LOGISTIC_DENSITY  # noqa: E402
from warp_sources import FUNNEL_THREAD_HAND, FUNNEL_WARP, FUNNEL_WARP_HAND, LOGISTIC_WARP  # noqa: E402

ab = r03.ab
TAPE_BYTES_CAP = r03.TAPE_BYTES_CAP


def warp_tape_traffic(nodes, d, Cn, es):
    """Bytes the warp-form tape moves in one gradient of Cn chains: each of the 32 lanes' nodes is recorded and swept
    as in the thread form (r03.tape_traffic); the chain's d input Vars (2 es bytes) are written once and q read once,
    and g is zeroed, then read and written back negated."""
    return Cn * (32 * nodes * ((8 + 3 * es) + (8 + 3 * es) + 4 * es) + d * (2 * es + es + es + 2 * es))


def tape_bytes(model, Cn):
    """Workspace bytes of the tape (8 + 3 * 8 bytes per node slot in FP64)."""
    slots = 32 * Cn if model.warp else (Cn + 31) // 32 * 32
    return model.tape_nodes * slots * 32


def gradient_row(model, form, density, d, Cn):
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
    ms, reps = r03.timed(call)
    model.check_tape()
    row = {"density": density, "form": form, "d": d, "chains": Cn, "ms_per_gradient": ms, "reps": reps,
           "window_s": ms * reps * 1e-3, "workspace_bytes": int(nbytes)}
    es = q.element_size()
    if model.reverse:
        tb = (warp_tape_traffic if model.warp else r03.tape_traffic)(model.tape_nodes, d, Cn, es)
        row.update({"tape_nodes_per_lane" if model.warp else "tape_nodes_per_chain": model.tape_nodes,
                    "tape_bytes_per_gradient": tb, "tape_gbs": tb / (ms * 1e-3) / 1e9,
                    "tape_frac_of_hbm_peak": tb / (ms * 1e-3) / 1e9 / r03.hbm_peak_gbs()})
    else:
        b = 2 * d * es * Cn
        row.update(bytes_per_gradient=b, gbs=b / (ms * 1e-3) / 1e9, frac_of_hbm_peak=b / (ms * 1e-3) / 1e9 /
                   r03.hbm_peak_gbs())
    return row


def make(form, src, d, data):
    if form == "thread-reverse":
        return r03.ReverseUserModel(src, d, data=data, autodiff=True)
    if form == "thread-hand":
        return ab.models.UserModel(src, d, data=data)
    return ab.models.UserModel(src, d, data=data, autodiff=form == "warp-reverse", warp=True)


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

    emit(dict(r03.gpu_info(), hbm_peak_gbs=r03.hbm_peak_gbs(), dtype="float64"))
    chains = (4096,) if a.quick else (4096, 65536)
    forms = {"funnel": (("thread-reverse", FUNNEL_DENSITY), ("warp-reverse", FUNNEL_WARP),
                        ("thread-hand", FUNNEL_THREAD_HAND), ("warp-hand", FUNNEL_WARP_HAND)),
             "logistic": (("thread-reverse", LOGISTIC_DENSITY), ("warp-reverse", LOGISTIC_WARP))}
    for density in ("funnel", "logistic"):
        for d in ((128,) if a.quick else (128, 1000, 4096)):
            data = r03.logistic_data(d) if density == "logistic" else None
            for form, src in forms[density]:
                model = make(form, src, d, data)
                for Cn in chains:
                    if model.reverse and tape_bytes(model, Cn) > TAPE_BYTES_CAP:
                        emit({"density": density, "form": form, "d": d, "chains": Cn, "skipped":
                              f"tape of {tape_bytes(model, Cn) / 1e9:.0f} GB", "tape_nodes": model.tape_nodes})
                        continue
                    emit(gradient_row(model, form, density, d, Cn))
                del model
                torch.cuda.empty_cache()
    d, Cn = (128, 512) if a.quick else (1000, 4096)
    for name, model in (("funnel thread-reverse", r03.ReverseUserModel(FUNNEL_DENSITY, d, autodiff=True)),
                        ("funnel warp-reverse", ab.models.UserModel(FUNNEL_WARP, d, autodiff=True, warp=True)),
                        ("funnel warp-hand", ab.models.UserModel(FUNNEL_WARP_HAND, d, warp=True)),
                        ("built-in NealFunnel", ab.models.NealFunnel(d))):
        emit(dict(r03.nuts_rate(model, d, Cn, 1 if a.quick else 3), model=name))


if __name__ == "__main__":
    main()
