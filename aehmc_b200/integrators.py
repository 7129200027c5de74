"""IntegratorState / velocity_verlet (reference integrators.py:7-75) over batched chains."""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple

import torch

from . import _lib, backend


class IntegratorState(NamedTuple):      # reference integrators.py:7-11
    position: torch.Tensor              # [C, d]
    momentum: torch.Tensor              # [C, d] or None
    potential_energy: torch.Tensor      # [C]
    potential_energy_grad: torch.Tensor # [C, d]


def new_integrator_state(potential_fn, position, momentum):
    """reference integrators.py:14-24; ``potential_fn`` is a model descriptor."""
    U, g = potential_fn.potential_and_grad(position)
    q = backend.as_device(position, potential_fn.dtype, potential_fn.device)
    return IntegratorState(q, momentum, U, g)


def velocity_verlet(potential_fn, kinetic_energy_fn):
    """reference integrators.py:27-75.  ``potential_fn``: model descriptor; ``kinetic_energy_fn``: the
    closure returned by ``gaussian_metric`` (it carries the metric).  The returned ``one_step(state,
    step_size)`` advances every chain by one fused kick-drift-kick; ``n_steps`` > 1 keeps the state
    on chip between steps (trajectory.static_integration)."""
    metric = kinetic_energy_fn.metric
    model = potential_fn
    lib = _lib.load()
    ws = backend.Workspace()

    def one_step(state, step_size, n_steps=1, direction=None):
        dev, dt = model.device, model.dtype
        q = state.position.clone()
        p = state.momentum.clone()
        U = state.potential_energy.clone()
        g = state.potential_energy_grad.clone()
        Cn = q.shape[0]
        eps = _per_chain(step_size, Cn, dev)
        dirs = None if direction is None else backend.as_device(direction, torch.int8, dev)
        m, mt = model.struct(), metric.struct()
        nbytes = lib.b2h_potential_workspace_bytes(C.byref(m), backend.code(dt), C.c_int64(Cn)) + q.numel() * 8 + 1024
        w = ws.get(nbytes, dev)
        _lib.check(lib.b2h_leapfrog(backend.context(dev), C.byref(m), C.byref(mt), backend.code(dt), backend.ptr(q),
                                    backend.ptr(p), backend.ptr(U), backend.ptr(g), backend.ptr(eps),
                                    backend.ptr(dirs), C.c_int32(n_steps), C.c_int64(Cn), backend.ptr(w),
                                    C.c_int64(w.numel())))
        model.check_tape()
        return IntegratorState(q, p, U, g)

    one_step.model = model
    one_step.metric = metric
    return one_step


def _per_chain(step_size, Cn, dev):
    """step size as float64 [C] on the device (scalar broadcasts)."""
    if isinstance(step_size, torch.Tensor):
        t = step_size.to(device=dev, dtype=torch.float64)
    else:
        t = torch.as_tensor(step_size, dtype=torch.float64, device=dev)
    if t.ndim == 0:
        t = t.expand(Cn)
    if t.shape != (Cn,):
        raise ValueError(f"step_size must be a scalar or [{Cn}]")
    return t.contiguous()
