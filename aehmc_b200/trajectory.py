"""Trajectory builders (reference trajectory.py).

``static_integration`` is the HMC inner loop.  The dynamic (NUTS) builders run inside the persistent
tick engine (csrc/engine.cuh): ``nuts.new_kernel`` drives whole transitions, and
``dynamic_integration`` / ``multiplicative_expansion`` below enter the same state machine with a
caller-supplied tree state (b2h_nuts_subtree / b2h_nuts_expand), one launch per call.
"""
from __future__ import annotations

from typing import NamedTuple

import ctypes as C

import torch

from . import _lib, backend
from .integrators import IntegratorState, _per_chain


class Diagnostics(NamedTuple):           # reference trajectory.py:379-384
    state: IntegratorState
    acceptance_probability: torch.Tensor  # [C] float64
    num_doublings: torch.Tensor           # [C] int32 (None for HMC)
    is_turning: torch.Tensor              # [C] bool  (None for HMC)
    is_diverging: torch.Tensor            # [C] bool


def static_integration(integrator, num_integration_steps):
    """reference trajectory.py:31-107: ``integrate(init_state, step_size) -> (state, updates)``.
    The whole fixed-length trajectory is one kernel launch."""

    def integrate(init_state, step_size):
        return integrator(init_state, step_size, n_steps=int(num_integration_steps)), {}

    return integrate


class MultiplicativeExpansionResult(NamedTuple):   # reference trajectory.py:387-393
    proposals: "ProposalState"
    right_states: IntegratorState
    left_states: IntegratorState
    momentum_sums: torch.Tensor
    termination_states: "TerminationState"
    diagnostics: Diagnostics


def _state_struct(st):
    return _lib.State(st.position.data_ptr(), st.momentum.data_ptr(), st.potential_energy_grad.data_ptr(),
                      st.potential_energy.data_ptr())


def _clone_state(st, dt, dev):
    return IntegratorState(backend.as_device(st.position, dt, dev).clone(),
                           backend.as_device(st.momentum, dt, dev).clone(),
                           backend.as_device(st.potential_energy, dt, dev).clone(),
                           backend.as_device(st.potential_energy_grad, dt, dev).clone())


def _tree_workspace(lib, ws, m, mt, cfg, Cn, dev):
    nbytes = lib.b2h_nuts_workspace_bytes(C.byref(m), C.byref(mt), C.byref(cfg), C.c_int64(Cn))
    if nbytes < 0:
        _lib.check(-1)
    return ws.get(nbytes, dev)


def dynamic_integration(srng, integrator, kinetic_energy, update_termination_state, is_criterion_met,
                        divergence_threshold, expansion=None, group=0):
    """reference trajectory.py:119-376.  ``integrator`` is the closure of ``velocity_verlet`` (it carries
    the model and the metric); the termination closures come from ``iterative_uturn`` and are
    accepted for signature parity -- the iterative U-turn criterion itself runs inside the engine.

    ``integrate(previous_last_state, direction, termination_state, max_num_steps, step_size,
    initial_energy)`` builds one sub-tree of ``1 + max_num_steps`` leapfrogs at most (SURVEY Q1) for
    every chain in ONE launch of the persistent kernel and returns ``((new_proposal, new_state,
    subtree_momentum_sum, new_termination_state, trajectory_length, is_diverging, has_terminated),
    updates)``.  The uniform draws of the in-tree progressive sampling are those of expansion
    ``expansion`` (default: log2(max_num_steps), its value inside NUTS) of the stream's current
    transition; the stream advances by one transition per call.  ``group``: threads per chain
    (0 = the engine's own choice)."""
    from .proposals import ProposalState
    from .termination import TerminationState

    model, metric = integrator.model, integrator.metric
    lib = _lib.load()
    ws = backend.Workspace()

    def integrate(previous_last_state, direction, termination_state, max_num_steps, step_size, initial_energy):
        dev, dt = model.device, model.dtype
        st = _clone_state(previous_last_state, dt, dev)
        Cn, d = st.position.shape
        maxd = int(termination_state.momentum_checkpoints.shape[1])
        n_steps = int(max_num_steps)
        k = expansion if expansion is not None else max(n_steps.bit_length() - 1, 0)
        dirs = backend.as_device(direction, torch.int8, dev).expand(Cn).contiguous()
        prop = IntegratorState(*[torch.empty_like(t) for t in st])
        energy = torch.empty(Cn, dtype=dt, device=dev)
        weight = torch.empty(Cn, dtype=torch.float64, device=dev)
        slpa = torch.empty(Cn, dtype=torch.float64, device=dev)
        msum = torch.empty_like(st.position)
        mck = backend.as_device(termination_state.momentum_checkpoints, dt, dev).clone()
        sck = backend.as_device(termination_state.momentum_sum_checkpoints, dt, dev).clone()
        imin = backend.as_device(termination_state.min_index, torch.int64, dev).clone()
        imax = backend.as_device(termination_state.max_index, torch.int64, dev).clone()
        E0 = backend.as_device(initial_energy, dt, dev).expand(Cn).contiguous()
        length = torch.empty(Cn, dtype=torch.int32, device=dev)
        div = torch.empty(Cn, dtype=torch.uint8, device=dev)
        term = torch.empty(Cn, dtype=torch.uint8, device=dev)
        eps = _per_chain(step_size, Cn, dev)
        sub = _lib.Subtree(_state_struct(st), dirs.data_ptr(), _state_struct(prop), energy.data_ptr(),
                           weight.data_ptr(), slpa.data_ptr(), msum.data_ptr(), mck.data_ptr(), sck.data_ptr(),
                           imin.data_ptr(), imax.data_ptr(), E0.data_ptr(), n_steps, int(k), length.data_ptr(),
                           div.data_ptr(), term.data_ptr())
        cfg = _lib.Cfg(backend.code(dt), maxd, float(divergence_threshold), 0, int(group), 0, 0, 0, 0)
        m, mt = model.struct(), metric.struct()
        rng, keep = srng.struct(1)
        w = _tree_workspace(lib, ws, m, mt, cfg, Cn, dev)
        _lib.check(lib.b2h_nuts_subtree(backend.context(dev), C.byref(m), C.byref(mt), C.byref(rng), C.byref(cfg),
                                        C.byref(sub), backend.ptr(eps), C.c_int64(Cn), backend.ptr(w),
                                        C.c_int64(w.numel())))
        model.check_tape()
        del keep
        srng.advance(1)
        return (ProposalState(prop, energy, weight, slpa), st, msum, TerminationState(mck, sck, imin, imax),
                length.to(torch.int64), div.bool(), term.bool()), {}

    integrate.model, integrate.metric = model, metric
    integrate.divergence_threshold = float(divergence_threshold)
    integrate.group = int(group)
    return integrate


def multiplicative_expansion(srng, trajectory_integrator, uturn_check_fn, max_num_expansions):
    """reference trajectory.py:396-714.  ``trajectory_integrator`` is the closure of
    ``dynamic_integration`` (it carries model, metric and divergence threshold).

    ``expand(proposal, left_state, right_state, momentum_sum, termination_state, initial_energy,
    step_size)`` runs the whole doubling loop of every chain in ONE launch.  The reference returns
    the scan history over expansions and its callers index ``[-1]`` (nuts.py:140-150); here every
    field has a leading axis of length 1 holding that final value."""
    from .proposals import ProposalState
    from .termination import TerminationState

    model, metric = trajectory_integrator.model, trajectory_integrator.metric
    thr = trajectory_integrator.divergence_threshold
    group = trajectory_integrator.group
    lib = _lib.load()
    ws = backend.Workspace()
    maxd = int(max_num_expansions)

    def expand(proposal, left_state, right_state, momentum_sum, termination_state, initial_energy, step_size):
        dev, dt = model.device, model.dtype
        prop = _clone_state(proposal.state, dt, dev)
        left = _clone_state(left_state, dt, dev)
        right = _clone_state(right_state, dt, dev)
        Cn, d = prop.position.shape
        if int(termination_state.momentum_checkpoints.shape[1]) != maxd:
            raise ValueError("termination state was not built for max_num_expansions")
        energy = backend.as_device(proposal.energy, dt, dev).expand(Cn).clone()
        weight = backend.as_device(proposal.weight, torch.float64, dev).expand(Cn).clone()
        slpa = backend.as_device(proposal.sum_log_p_accept, torch.float64, dev).expand(Cn).clone()
        msum = backend.as_device(momentum_sum, dt, dev).clone()
        mck = backend.as_device(termination_state.momentum_checkpoints, dt, dev).clone()
        sck = backend.as_device(termination_state.momentum_sum_checkpoints, dt, dev).clone()
        imin = backend.as_device(termination_state.min_index, torch.int64, dev).clone()
        imax = backend.as_device(termination_state.max_index, torch.int64, dev).clone()
        E0 = backend.as_device(initial_energy, dt, dev).expand(Cn).contiguous()
        eps = _per_chain(step_size, Cn, dev)
        acc = torch.empty(Cn, dtype=torch.float64, device=dev)
        nd = torch.zeros(Cn, dtype=torch.int32, device=dev)
        turning = torch.zeros(Cn, dtype=torch.uint8, device=dev)
        diverging = torch.zeros(Cn, dtype=torch.uint8, device=dev)
        nleap = torch.zeros(Cn, dtype=torch.int32, device=dev)
        diag = _lib.Diag(acc.data_ptr(), nd.data_ptr(), turning.data_ptr(), diverging.data_ptr(), nleap.data_ptr())
        tree = _lib.Tree(_state_struct(prop), energy.data_ptr(), weight.data_ptr(), slpa.data_ptr(),
                         _state_struct(left), _state_struct(right), msum.data_ptr(), mck.data_ptr(), sck.data_ptr(),
                         imin.data_ptr(), imax.data_ptr(), E0.data_ptr())
        cfg = _lib.Cfg(backend.code(dt), maxd, thr, 0, group, 0, 0, 0, 0)
        m, mt = model.struct(), metric.struct()
        rng, keep = srng.struct(1)
        w = _tree_workspace(lib, ws, m, mt, cfg, Cn, dev)
        _lib.check(lib.b2h_nuts_expand(backend.context(dev), C.byref(m), C.byref(mt), C.byref(rng), C.byref(cfg),
                                       C.byref(tree), backend.ptr(eps), C.c_int64(Cn), C.byref(diag), backend.ptr(w),
                                       C.c_int64(w.numel())))
        model.check_tape()
        del keep
        srng.advance(1)
        h = lambda t: t.unsqueeze(0)
        hs = lambda s: IntegratorState(*[h(t) for t in s])
        result = MultiplicativeExpansionResult(
            proposals=ProposalState(hs(prop), h(energy), h(weight), h(slpa)),
            right_states=hs(right), left_states=hs(left), momentum_sums=h(msum),
            termination_states=TerminationState(h(mck), h(sck), h(imin), h(imax)),
            diagnostics=Diagnostics(hs(prop), h(acc), h(nd.to(torch.int64)), h(turning.bool()), h(diverging.bool())))
        return result, {}

    return expand


def where_proposal(do_pick_left, left_proposal, right_proposal):
    """reference trajectory.py:717-735: per-chain switch between two proposals."""
    from .proposals import ProposalState, _select

    dev = left_proposal.weight.device
    Cn = left_proposal.weight.shape[0]
    mask = backend.as_device(do_pick_left, torch.uint8, dev).expand(Cn).contiguous()
    st = IntegratorState(*[_select(mask, a, b) for a, b in zip(left_proposal.state, right_proposal.state)])
    return ProposalState(st, _select(mask, left_proposal.energy, right_proposal.energy),
                         _select(mask, left_proposal.weight, right_proposal.weight),
                         _select(mask, left_proposal.sum_log_p_accept, right_proposal.sum_log_p_accept))
