"""Stan-style window adaptation (reference window_adaptation.py) for many chains.

Every chain adapts its own step size (dual averaging) and diagonal or, with ``is_mass_matrix_full``, dense
inverse mass matrix (Welford), exactly as running the reference once per chain would.  ``run`` executes the whole warm-up on the
device inside the tick engine when ``kernel`` comes from ``nuts.new_kernel`` / ``hmc.new_kernel``;
``window_adaptation(...) -> (init, update)`` is the composable form built on the batched
adaptation primitives.
"""
from __future__ import annotations

from typing import List, Tuple

import torch

from . import _engine, _lib, backend, metrics
from .integrators import IntegratorState
from .mass_matrix import covariance_adaptation
from .step_size import dual_averaging_adaptation


def build_schedule(num_steps: int, initial_buffer_size: int = 75, final_buffer_size: int = 50,
                   first_window_size: int = 25) -> List[Tuple[int, bool]]:
    """Host-side schedule, same contract as reference window_adaptation.py:230-327:
    [(stage, is_middle_window_end)] with stage 0 = fast (step size only), 1 = slow."""
    if num_steps < 20:
        return [(0, False)] * num_steps
    if initial_buffer_size + first_window_size + final_buffer_size > num_steps:
        initial_buffer_size = int(0.15 * num_steps)
        final_buffer_size = int(0.1 * num_steps)
        first_window_size = num_steps - initial_buffer_size - final_buffer_size
    slow_end = num_steps - final_buffer_size
    ends = set()
    start, size = initial_buffer_size, first_window_size
    while start < slow_end:
        width = size
        if 3 * size <= slow_end - start:
            size *= 2
        else:
            width = slow_end - start
        start += width
        ends.add(start - 1)
    return [(1 if initial_buffer_size <= i < slow_end else 0, i in ends) for i in range(num_steps)]


def run(kernel, initial_state: IntegratorState, num_steps=1000, *, is_mass_matrix_full=False,
        initial_step_size=1.0, target_acceptance_rate=0.80, num_integration_steps=None, pooled=False,
        max_chunk_bytes=2 << 30, initial_inverse_mass_matrix=None):
    """reference window_adaptation.py:17-116 -> (last_chain_state, (step_size[C], imm[C, d]), updates).

    ``is_mass_matrix_full=True`` adapts one dense matrix per chain (d <= 128) and returns imm[C, d, d]; sample with
    ``metrics.per_chain(imm)``.

    ``pooled=True`` (not in the reference, which adapts one chain at a time): the chains sample the same target, so
    the inverse mass matrix is ONE matrix -- diagonal [d] or, with ``is_mass_matrix_full``, dense [d, d] -- estimated
    at each slow-window end from the positions of all chains of all ranks (Welford states merged over NCCL); step
    sizes stay per chain.  ``initial_inverse_mass_matrix`` (pooled mode only; the reference always starts from the
    identity) is the metric used until the first window end.  Returns (state, (step_size[C], imm[d] or imm[d, d]),
    updates)."""
    spec = getattr(kernel, "spec", None)
    if pooled:
        if spec is None:
            raise ValueError("pooled warm-up needs a kernel from nuts.new_kernel / hmc.new_kernel")
        return _run_pooled(spec, initial_state, num_steps, is_mass_matrix_full, initial_step_size,
                           target_acceptance_rate, num_integration_steps, max_chunk_bytes, initial_inverse_mass_matrix)
    if initial_inverse_mass_matrix is not None:
        raise ValueError("initial_inverse_mass_matrix needs pooled=True (per-chain warm-up starts from the identity)")
    Cn, d = initial_state.position.shape
    if spec is not None and is_mass_matrix_full and Cn > 1:
        return _run_per_chain_dense(spec, initial_state, num_steps, initial_step_size, target_acceptance_rate,
                                    num_integration_steps, max_chunk_bytes)
    if spec is None or is_mass_matrix_full:
        return _run_composed(kernel, initial_state, num_steps, is_mass_matrix_full, initial_step_size,
                             target_acceptance_rate, num_integration_steps)
    model = spec["model"]
    schedule = build_schedule(num_steps)
    adapt = _engine.AdaptState(Cn, schedule, model.device, target_acceptance_rate, float(initial_step_size))
    imm = metrics.GaussianMetric(metrics.per_chain(torch.ones((Cn, d), dtype=model.dtype, device=model.device)))
    kw = dict(n_transitions=num_steps, divergence_threshold=spec["divergence_threshold"], adapt=adapt)
    if spec["kind"] == "nuts":
        kw["max_num_expansions"] = spec["max_num_expansions"]
        kw["exact_doubling"] = spec.get("exact_doubling", False)
    else:
        if num_integration_steps is None:
            raise ValueError("HMC warm-up needs num_integration_steps")
        kw["num_integration_steps"] = num_integration_steps
    info, extras = _engine.run(spec["kind"], model, imm, spec["srng"], initial_state, 1.0, **kw)
    st = info.state
    last = IntegratorState(st.position, None, st.potential_energy, st.potential_energy_grad)
    return last, (extras["step_size"], imm.imm), {"n_leapfrog": extras["n_leapfrog"]}


def window_adaptation(num_steps, is_mass_matrix_full=False, initial_step_size=1.0, target_acceptance_rate=0.80):
    """reference window_adaptation.py:119-227 -> (init(state), update(step, warmup_state, parameters, chain_info))."""
    mm_init, mm_update, mm_final = covariance_adaptation(is_mass_matrix_full)
    da_init, da_update = dual_averaging_adaptation(target_acceptance_rate)
    schedule = build_schedule(num_steps)

    def init(initial_chain_state):
        q = initial_chain_state.position
        Cn, d = q.shape
        imm, mm_state = mm_init(d, Cn, q.dtype, q.device)
        da_state = da_init(torch.full((Cn,), float(initial_step_size), dtype=torch.float64, device=q.device))
        return (da_state, mm_state), (torch.exp(da_state.iterates), imm)

    def update(step, warmup_state, parameters, chain_info):
        da_state, mm_state = warmup_state
        stage, is_middle_window_end = schedule[step]
        da_state = da_update(chain_info.acceptance_probability, da_state)
        if stage == 1:
            mm_state = mm_update(chain_info.state.position, mm_state)
        step_size, imm = torch.exp(da_state.iterates), parameters[1]
        if is_middle_window_end:                                    # slow_final (:165-190)
            imm = mm_final(mm_state)
            Cn, d = chain_info.state.position.shape
            _, mm_state = mm_init(d, Cn, imm.dtype, imm.device)
            da_state = da_init(step_size)
        if step == num_steps - 1:
            step_size = torch.exp(da_state.iterates_avg)
        return (da_state, mm_state), (step_size, imm)

    return init, update


def _run_composed(kernel, initial_state, num_steps, is_mass_matrix_full, initial_step_size, target,
                  num_integration_steps=None):
    init_adapt, update_adapt = window_adaptation(num_steps, is_mass_matrix_full, initial_step_size, target)
    warmup_state, parameters = init_adapt(initial_state)
    Cn = initial_state.position.shape[0]
    spec = getattr(kernel, "spec", None)
    is_hmc = (spec is not None and spec.get("kind") == "hmc") or (spec is None and num_integration_steps is not None)
    if is_hmc and num_integration_steps is None:
        raise ValueError("HMC warm-up needs num_integration_steps")
    state = initial_state
    for step in range(num_steps):
        step_size, imm = parameters
        arg = imm[0] if is_mass_matrix_full and Cn == 1 else metrics.per_chain(imm)
        if is_hmc:
            info, _ = kernel(state, step_size, arg, num_integration_steps)
        else:
            info, _ = kernel(state, step_size, arg)
        warmup_state, parameters = update_adapt(step, warmup_state, parameters, info)
        s = info.state
        state = IntegratorState(s.position, None, s.potential_energy, s.potential_energy_grad)
    return state, parameters, {}


def _engine_kw(spec, adapt, num_integration_steps):
    kw = dict(divergence_threshold=spec["divergence_threshold"], adapt=adapt)
    if spec["kind"] == "nuts":
        kw["max_num_expansions"] = spec["max_num_expansions"]
        kw["exact_doubling"] = spec.get("exact_doubling", False)
    else:
        if num_integration_steps is None:
            raise ValueError("HMC warm-up needs num_integration_steps")
        kw["num_integration_steps"] = num_integration_steps
    return kw


def _run_windows(spec, initial_state, schedule, imm, metric_of, stats, kw, max_chunk_bytes):
    """The warm-up in chunks that end at window ends.  The engine runs the transitions of a chunk (per-chain dual
    averaging on the device, window_adaptation.py:194-215); between chunks the draws of the slow stage are folded into
    ``stats``, and at a window end (window_adaptation.py:165-190) ``stats.final`` gives the new inverse mass matrix,
    which ``metric_of`` turns into what the engine samples with."""
    model = spec["model"]
    dt = model.dtype
    Cn, d = initial_state.position.shape
    num_steps = len(schedule)
    adapt = kw["adapt"]
    chunk_max = max(1, int(max_chunk_bytes) // max(Cn * d * initial_state.position.element_size(), 1))
    state, eps, step, n_leap = initial_state, 1.0, 0, None
    metric = metric_of(imm)
    windows = []
    while step < num_steps:
        end = step
        while end < num_steps - 1 and not schedule[end][1] and end - step + 1 < chunk_max:
            end += 1
        n = end - step + 1
        slow = [i - step for i in range(step, end + 1) if schedule[i][0] == 1]
        adapt.step_offset = step
        info, extras = _engine.run(spec["kind"], model, metric, spec["srng"], state, eps, n_transitions=n,
                                   store_draws=n if slow else 0, **kw)
        eps = extras["step_size"]
        if slow:
            stats.update(extras["draws"][slow[0]:slow[-1] + 1])          # the slow stage is one contiguous range
        if schedule[end][1]:
            stats.all_reduce()
            windows.append(stats.n)
            imm = stats.final(dt)
            metric = metric_of(imm)
            stats.reset()
        st = info.state
        state = IntegratorState(st.position, None, st.potential_energy, st.potential_energy_grad)
        n_leap = extras["n_leapfrog"]
        step = end + 1
    return state, eps, imm, n_leap, windows


def _run_pooled(spec, initial_state, num_steps, is_mass_matrix_full, initial_step_size, target, num_integration_steps,
                max_chunk_bytes, initial_imm=None):
    """Warm-up with cross-chain statistics: the draws of the slow stage go into the pooled Welford state, and at a
    window end the per-rank states are merged over the process group and every rank rebuilds the same shared
    metric."""
    from .mass_matrix import PooledWelford
    model = spec["model"]
    dev, dt = model.device, model.dtype
    Cn, d = initial_state.position.shape
    schedule = build_schedule(num_steps)
    adapt = _engine.AdaptState(Cn, schedule, dev, target, float(initial_step_size), pooled=True)
    imm = torch.eye(d, dtype=dt, device=dev) if is_mass_matrix_full else torch.ones(d, dtype=dt, device=dev)
    if initial_imm is not None:
        imm0 = backend.as_device(initial_imm, dt, dev)
        if imm0.shape != imm.shape:
            raise ValueError(f"initial_inverse_mass_matrix must have shape {tuple(imm.shape)}")
        imm = imm0
    pool = PooledWelford(d, is_mass_matrix_full, dev)
    kw = _engine_kw(spec, adapt, num_integration_steps)
    state, eps, imm, n_leap, windows = _run_windows(spec, initial_state, schedule, imm, lambda m: m, pool, kw,
                                                    max_chunk_bytes)
    return state, (eps, imm), {"n_leapfrog": n_leap, "pooled_window_sizes": windows}


def _run_per_chain_dense(spec, initial_state, num_steps, initial_step_size, target, num_integration_steps,
                         max_chunk_bytes):
    """Per-chain dense warm-up: what the reference's ``is_mass_matrix_full=True`` does for one chain, for every chain.
    The engine runs the dual averaging (pooled mode: it never touches the metric); each chain's slow-stage draws are
    folded into its own Welford state in transition order, and at a window end every chain's matrix is rebuilt and
    refactored on the device."""
    from .mass_matrix import PerChainWelford
    model = spec["model"]
    dev, dt = model.device, model.dtype
    Cn, d = initial_state.position.shape
    if d > _lib.DENSE_PER_CHAIN_MAX_DIM:
        raise ValueError(f"per-chain dense adaptation needs dim <= {_lib.DENSE_PER_CHAIN_MAX_DIM}, got {d}; adapt one "
                         "shared dense matrix instead (pooled=True)")
    schedule = build_schedule(num_steps)
    adapt = _engine.AdaptState(Cn, schedule, dev, target, float(initial_step_size), pooled=True)
    imm = torch.eye(d, dtype=dt, device=dev).expand(Cn, d, d).contiguous()
    kw = _engine_kw(spec, adapt, num_integration_steps)
    metric_of = lambda m: metrics.GaussianMetric(metrics.per_chain(m), dt, dev)
    state, eps, imm, n_leap, _ = _run_windows(spec, initial_state, schedule, imm, metric_of,
                                              PerChainWelford(Cn, d, dt, dev), kw, max_chunk_bytes)
    return state, (eps, imm), {"n_leapfrog": n_leap}
