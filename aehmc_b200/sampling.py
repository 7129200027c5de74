"""Many transitions per call (the reference drives ``kernel`` from an outer ``aesara.scan``,
e.g. reference tests/test_hmc.py:296-324; here the loop stays on the device), thinned draw storage and the
checkpoint / resume format of a run (SURVEY 8f row 4)."""
from __future__ import annotations

import torch

from . import _engine, _lib, metrics
from .integrators import IntegratorState
from .random import RandomStream

CHECKPOINT_VERSION = 2
# "per_chain" covers the diagonal [C, d] and the dense [C, d, d] kinds: the shape tells them apart
_KIND_NAMES = {_lib.IMM_SCALAR: "scalar", _lib.IMM_DIAG: "diag", _lib.IMM_DIAG_PER_CHAIN: "per_chain",
               _lib.IMM_DENSE: "dense", _lib.IMM_DENSE_PER_CHAIN: "per_chain"}


def sample(kernel, state, step_size, inverse_mass_matrix, num_samples, *, num_integration_steps=None,
           store_draws=True, group=0, thin=1):
    """Run ``num_samples`` transitions of every chain.  Returns (Diagnostics of the last transition,
    draws [ceil(num_samples / thin), C, d] or None, stats [same, C, 4], extras): slot k holds transition k * thin."""
    spec = kernel.spec
    thin = max(int(thin), 1)
    n_slots = (num_samples + thin - 1) // thin
    kw = dict(n_transitions=num_samples, divergence_threshold=spec["divergence_threshold"],
              store_draws=n_slots if store_draws else 0, group=group, thin=thin)
    if spec["kind"] == "nuts":
        kw["max_num_expansions"] = spec["max_num_expansions"]
        kw["exact_doubling"] = spec.get("exact_doubling", False)
    else:
        kw["num_integration_steps"] = int(num_integration_steps)
    info, extras = _engine.run(spec["kind"], spec["model"], inverse_mass_matrix, spec["srng"], state, step_size, **kw)
    return info, extras["draws"], extras["draw_stats"], extras


def checkpoint(state, srng, step_size, inverse_mass_matrix):
    """Everything needed to continue a run bit-for-bit: the chain state, the step size(s), the inverse mass matrix
    and the Philox coordinates (seed, global chain offset, transition counter).  A plain dict of CPU tensors and
    ints: ``torch.save`` / ``torch.load`` is the wire format.  Draws are a pure function of (seed, chain id,
    transition), so the continuation equals the uninterrupted run on any number of GPUs."""
    if not isinstance(srng, RandomStream):
        raise TypeError("only RandomStream runs can be checkpointed (injected draws are consumed from transition 0)")
    def cpu(t):
        if t is None:
            return None
        if not isinstance(t, torch.Tensor):          # Python floats / NumPy arrays: keep float64 (0.3 must stay 0.3)
            import numpy as np
            t = torch.from_numpy(np.asarray(t, dtype=np.float64).copy())
        return t.detach().to("cpu").clone()

    # the inverse mass matrix keeps its kind: a [C, d] per-chain diagonal (what window adaptation returns) must not
    # come back as a dense [d, d] matrix
    imm = inverse_mass_matrix
    if isinstance(imm, metrics.GaussianMetric):
        kind = _KIND_NAMES[imm.kind]
        imm = torch.tensor(imm.scalar, dtype=torch.float64) if kind == "scalar" else imm.imm
    elif isinstance(imm, metrics.per_chain):
        kind, imm = "per_chain", imm.imm
    else:
        imm = cpu(imm)
        if imm.ndim > 2:
            raise ValueError(f"Expected a mass matrix of dimension 1 (diagonal) or 2, got {imm.ndim}")
        kind = ("scalar", "diag", "dense")[imm.ndim]
    return {"version": CHECKPOINT_VERSION,
            "position": cpu(state.position), "potential_energy": cpu(state.potential_energy),
            "potential_energy_grad": cpu(state.potential_energy_grad),
            "step_size": cpu(step_size), "inverse_mass_matrix": cpu(imm), "inverse_mass_matrix_kind": kind,
            "seed": srng.seed, "chain_offset": srng.chain_offset, "transition": srng.transition}


def restore(ckpt, device=None):
    """Inverse of :func:`checkpoint`: returns (state, srng, step_size, inverse_mass_matrix) on ``device``; a
    per-chain inverse mass matrix (diagonal [C, d] or dense [C, d, d]) comes back wrapped in ``metrics.per_chain``."""
    if ckpt.get("version") != CHECKPOINT_VERSION:
        raise ValueError(f"unknown checkpoint version {ckpt.get('version')}")
    dev = torch.device("cuda" if device is None else device)
    up = lambda t: None if t is None else t.to(dev)
    state = IntegratorState(up(ckpt["position"]), None, up(ckpt["potential_energy"]), up(ckpt["potential_energy_grad"]))
    srng = RandomStream(ckpt["seed"], ckpt["chain_offset"])
    srng.transition = int(ckpt["transition"])
    imm = up(ckpt["inverse_mass_matrix"])
    if ckpt["inverse_mass_matrix_kind"] == "per_chain":
        imm = metrics.per_chain(imm)
    return state, srng, up(ckpt["step_size"]), imm
