"""Python side of b2h_nuts_run / b2h_hmc_run: argument marshalling only."""
from __future__ import annotations

import ctypes as C
import weakref

import torch

from . import _lib, backend
from .integrators import IntegratorState, _per_chain
from .metrics import GaussianMetric
from .trajectory import Diagnostics

_workspaces = {}
_resume_offsets = {}
_resume_groups = {}


def _evict(key):
    _workspaces.pop(key, None)
    _resume_offsets.pop(key, None)
    _resume_groups.pop(key, None)


def _workspace(key, nbytes, dev, owner=None):
    """Engine workspace of one (model, chain count): freed with the model that owns it (an explicit
    ``workspace_key`` lives until ``release_workspace(key)``)."""
    ws = _workspaces.get(key)
    if ws is None:
        ws = _workspaces[key] = backend.Workspace()
        if owner is not None:
            try:
                weakref.finalize(owner, _evict, key)
            except TypeError:
                pass
    return ws.get(nbytes, dev)


def release_workspace(key):
    """Drop the workspace (and the chain state machines kept in it) of an explicit ``workspace_key``."""
    _evict(key)


class AdaptState:
    """Device arrays of the per-chain warm-up state (b2h_adapt)."""

    def __init__(self, Cn, schedule, dev, target=0.8, initial_step_size=1.0, gamma=0.05, t0=10, kappa=0.75,
                 pooled=False):
        self.pooled, self.step_offset = bool(pooled), 0
        self.num_steps = len(schedule)
        self.stage = torch.tensor([s for s, _ in schedule], dtype=torch.uint8, device=dev)
        self.window_end = torch.tensor([1 if e else 0 for _, e in schedule], dtype=torch.uint8, device=dev)
        self.target, self.gamma, self.t0, self.kappa = float(target), float(gamma), float(t0), float(kappa)
        self.initial_step_size = float(initial_step_size)
        self.da_step = torch.ones(Cn, dtype=torch.int64, device=dev)
        self.da_x = torch.zeros(Cn, dtype=torch.float64, device=dev)
        self.da_x_avg = torch.zeros(Cn, dtype=torch.float64, device=dev)
        self.da_g_avg = torch.zeros(Cn, dtype=torch.float64, device=dev)
        self.da_mu = torch.full((Cn,), float(initial_step_size), dtype=torch.float64, device=dev)
        self.wc_n = torch.zeros(Cn, dtype=torch.int64, device=dev)

    def struct(self):
        return _lib.Adapt(1, self.num_steps, self.stage.data_ptr(), self.window_end.data_ptr(), self.target,
                          self.gamma, self.t0, self.kappa, self.initial_step_size, self.da_step.data_ptr(),
                          self.da_x.data_ptr(), self.da_x_avg.data_ptr(), self.da_g_avg.data_ptr(),
                          self.da_mu.data_ptr(), None, None, self.wc_n.data_ptr(), 1 if self.pooled else 0,
                          int(self.step_offset))


def run(kind, model, metric, srng, state, step_size, *, n_transitions=1, max_num_expansions=10,
        divergence_threshold=1000.0, num_integration_steps=0, adapt=None, store_draws=0, max_ticks=0,
        resume=False, group=0, workspace_key=None, return_counters=False, thin=1, exact_doubling=False):
    """Run ``n_transitions`` HMC/NUTS transitions of every chain (or ``max_ticks`` leapfrog ticks).
    ``store_draws`` slots are filled with every ``thin``-th transition of the call (slot k = transition k * thin).
    Returns (Diagnostics of the last transition, extras dict)."""
    lib = _lib.load()
    dev, dt = model.device, model.dtype
    metric = metric if isinstance(metric, GaussianMetric) else GaussianMetric(metric, dt, dev)
    if metric.dtype != dt:
        raise ValueError("metric and model dtypes differ")
    q = backend.as_device(state.position, dt, dev).clone()
    if q.ndim != 2 or q.shape[1] != model.dim:
        raise ValueError(f"position must be [chains, {model.dim}]")
    Cn, d = q.shape
    if metric.dim is not None and metric.dim != d:
        raise ValueError("inverse mass matrix and position dimensions differ")
    if metric.kind == _lib.IMM_DIAG_PER_CHAIN and metric.imm.shape[0] != Cn:
        raise ValueError("per-chain inverse mass matrix must be [chains, dim]")
    if metric.kind == _lib.IMM_DENSE_PER_CHAIN and tuple(metric.imm.shape) != (Cn, d, d):
        raise ValueError(f"per-chain dense inverse mass matrix must be [chains, dim, dim] = [{Cn}, {d}, {d}], got "
                         f"{list(metric.imm.shape)}")
    U = backend.as_device(state.potential_energy, dt, dev).clone()
    g = backend.as_device(state.potential_energy_grad, dt, dev).clone()
    p = torch.empty_like(q)
    eps = _per_chain(step_size, Cn, dev).clone()
    cfg = _lib.Cfg(backend.code(dt), int(max_num_expansions), float(divergence_threshold),
                   int(num_integration_steps), int(group), 0, int(thin), 1 if exact_doubling else 0, 0)
    m, mt = model.struct(), metric.struct()
    rng, keep = srng.struct(n_transitions)
    acc = torch.empty(Cn, dtype=torch.float64, device=dev)
    nd = torch.zeros(Cn, dtype=torch.int32, device=dev)
    turning = torch.zeros(Cn, dtype=torch.uint8, device=dev)
    diverging = torch.zeros(Cn, dtype=torch.uint8, device=dev)
    nleap = torch.zeros(Cn, dtype=torch.int32, device=dev)
    diag = _lib.Diag(acc.data_ptr(), nd.data_ptr(), turning.data_ptr(), diverging.data_ptr(), nleap.data_ptr())
    draws = stats = None
    if store_draws > 0:
        draws = torch.empty((store_draws, Cn, d), dtype=dt, device=dev)
        stats = torch.empty((store_draws, Cn, 4), dtype=torch.float64, device=dev)
    counters = torch.zeros(4, dtype=torch.int64, device=dev)
    nbytes = lib.b2h_nuts_workspace_bytes(C.byref(m), C.byref(mt), C.byref(cfg), C.c_int64(Cn))
    if nbytes < 0:
        _lib.check(-1)
    key = workspace_key or (kind, id(model), Cn, dev.index)
    ws = _workspace(key, nbytes, dev, owner=None if workspace_key else model)
    # a resumed call continues the transitions in flight: it keeps the Philox transition offset of the call that
    # started the run (the chain records count transitions cumulatively), so draws stay a pure function of
    # (seed, chain, transition) however the run is chunked
    if resume and key in _resume_offsets:
        rng.transition_offset = _resume_offsets[key]
        cfg.group = _resume_groups[key]          # the workspace layout is the one of the call that started the run
    else:
        _resume_offsets[key] = int(rng.transition_offset)
        _resume_groups[key] = int(lib.b2h_nuts_plan_group(C.byref(m), C.byref(mt), C.byref(cfg), C.c_int64(Cn),
                                                          C.c_int32(1 if max_ticks > 0 else 0)))
    ad = adapt.struct() if adapt is not None else None
    ctx = backend.context(dev)
    if kind == "nuts":
        rc = lib.b2h_nuts_run(ctx, C.byref(m), C.byref(mt), C.byref(rng), C.byref(cfg),
                              C.byref(ad) if ad is not None else None, backend.ptr(q), backend.ptr(p),
                              backend.ptr(U), backend.ptr(g), backend.ptr(eps), C.c_int64(Cn),
                              C.c_int32(n_transitions), C.c_int64(max_ticks), C.c_int32(1 if resume else 0),
                              C.byref(diag), backend.ptr(draws), backend.ptr(stats), C.c_int32(store_draws),
                              backend.ptr(counters), backend.ptr(ws), C.c_int64(ws.numel()))
    else:
        rc = lib.b2h_hmc_run(ctx, C.byref(m), C.byref(mt), C.byref(rng), C.byref(cfg),
                             C.byref(ad) if ad is not None else None, backend.ptr(q), backend.ptr(p),
                             backend.ptr(U), backend.ptr(g), backend.ptr(eps), C.c_int64(Cn),
                             C.c_int32(n_transitions), C.byref(diag), backend.ptr(draws), backend.ptr(stats),
                             C.c_int32(store_draws), backend.ptr(counters), backend.ptr(ws), C.c_int64(ws.numel()))
    _lib.check(rc)
    model.check_tape()
    del keep
    srng.advance(n_transitions)
    new_state = IntegratorState(q, p, U, g)
    if kind == "nuts":
        info = Diagnostics(new_state, acc, nd, turning.bool(), diverging.bool())
    else:
        info = Diagnostics(new_state, acc, None, None, diverging.bool())
    extras = {"n_leapfrog": nleap, "step_size": eps, "draws": draws, "draw_stats": stats,
              "inverse_mass_matrix": metric.imm if metric.kind == _lib.IMM_DIAG_PER_CHAIN else None}
    if return_counters:
        extras["counters"] = counters
    return info, extras
