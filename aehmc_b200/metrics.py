"""gaussian_metric (reference metrics.py:10-106) over batched chains.

``gaussian_metric(inverse_mass_matrix)`` keeps the reference's contract: a 0-d, 1-d (diagonal)
or 2-d (dense, shared by all chains) inverse mass matrix, ``ValueError`` above 2-d, and returns
``(momentum_generator, kinetic_energy, is_turning)``.  One matrix per chain (what per-chain window
adaptation produces) is passed as ``per_chain(imm[C, d])`` (diagonal) or ``per_chain(imm[C, d, d])`` (dense).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib, backend


class per_chain:
    """Marks a tensor as one inverse mass matrix per chain: ``[chains, dim]`` diagonal or ``[chains, dim, dim]``
    dense (dim <= 128).  A dense one is symmetrised, ``(A + A^T) / 2`` as for a shared matrix, and factored on the
    device (``b2h_dense_factor_per_chain``, FP64 Cholesky); ``ValueError`` names the chains whose matrix is not
    positive definite."""

    def __init__(self, imm):
        self.imm = imm


class GaussianMetric:
    def __init__(self, inverse_mass_matrix, dtype=None, device=None):
        imm = inverse_mass_matrix
        if isinstance(imm, GaussianMetric):
            self.__dict__.update(imm.__dict__)
            return
        pc = isinstance(imm, per_chain)
        if pc:
            imm = imm.imm
        if isinstance(imm, torch.Tensor):
            dtype = dtype or imm.dtype
            device = device or (imm.device if imm.is_cuda else None)
        self.dtype = backend.torch_dtype(dtype or torch.float64)
        self.device = backend.device(device)
        ndim = imm.ndim if isinstance(imm, torch.Tensor) else np.ndim(imm)
        self.scalar, self.imm, self.sqrt_t, self.chol_t = 0.0, None, None, None
        if pc and ndim == 3:
            self._factor_per_chain(backend.as_device(imm, self.dtype, self.device))
        elif pc:
            if ndim != 2:
                raise ValueError("per_chain() expects a [chains, dim] or [chains, dim, dim] tensor")
            self.kind = _lib.IMM_DIAG_PER_CHAIN
            self.imm = backend.as_device(imm, self.dtype, self.device)
            self.dim = int(self.imm.shape[1])
        elif ndim == 0:
            self.kind, self.dim = _lib.IMM_SCALAR, None
            self.scalar = float(imm)
        elif ndim == 1:
            self.kind = _lib.IMM_DIAG
            self.imm = backend.as_device(imm, self.dtype, self.device)
            self.dim = int(self.imm.numel())
        elif ndim == 2:
            # reference metrics.py:52-59: L = chol(imm), mass_matrix_sqrt = solve_triangular(L, I, lower, trans).
            # One-off host factorisation (the reference rebuilds it inside every call).
            import scipy.linalg
            a = np.asarray(imm.detach().cpu() if isinstance(imm, torch.Tensor) else imm, dtype=np.float64)
            a = 0.5 * (a + a.T)     # dK/dp of 0.5 p^T A p uses the symmetric part (integrators.py:61)
            L = np.linalg.cholesky(a)
            sqrt = scipy.linalg.solve_triangular(L, np.eye(a.shape[0]), lower=True, trans="T")
            self.kind = _lib.IMM_DENSE
            self.imm = backend.as_device(a, self.dtype, self.device)
            self.sqrt_t = backend.as_device(np.ascontiguousarray(sqrt.T), self.dtype, self.device)
            # imm . (L^-T z) = L z: the engine draws a transition's momentum and its velocity from the same normals
            self.chol_t = backend.as_device(np.ascontiguousarray(L.T), self.dtype, self.device)
            self.dim = int(a.shape[0])
        else:
            raise ValueError(f"Expected a mass matrix of dimension 1 (diagonal) or 2, got {ndim}")
        self._ws = backend.Workspace()

    def _factor_per_chain(self, a):
        Cn, d, d2 = a.shape
        if d != d2:
            raise ValueError(f"per_chain() dense matrices must be square, got [{Cn}, {d}, {d2}]")
        if not 1 <= d <= _lib.DENSE_PER_CHAIN_MAX_DIM:
            raise ValueError(f"per-chain dense inverse mass matrices need dim <= {_lib.DENSE_PER_CHAIN_MAX_DIM}, got "
                             f"{d}; adapt one shared dense matrix instead (window_adaptation.run(..., pooled=True))")
        self.kind, self.dim = _lib.IMM_DENSE_PER_CHAIN, int(d)
        self.imm, self.sqrt_t, self.chol_t = (torch.empty_like(a) for _ in range(3))
        info = torch.empty(Cn, dtype=torch.int32, device=self.device)
        _lib.check(_lib.load().b2h_dense_factor_per_chain(
            backend.context(self.device), backend.code(self.dtype), backend.ptr(a), backend.ptr(self.imm),
            backend.ptr(self.sqrt_t), backend.ptr(self.chol_t), backend.ptr(info), C.c_int64(Cn), C.c_int64(d)))
        bad = torch.nonzero(info).flatten().tolist()
        if bad:
            shown = ", ".join(str(c) for c in bad[:8]) + (f" and {len(bad) - 8} more" if len(bad) > 8 else "")
            raise ValueError(f"per_chain(): the inverse mass matrix is not positive definite for chain(s) {shown}")

    def struct(self):
        p = lambda t: None if t is None else t.data_ptr()
        # flags bit 0: sqrt_t / chol_t are the triangular Cholesky factors built here (b200hmc.h)
        dense = self.kind in (_lib.IMM_DENSE, _lib.IMM_DENSE_PER_CHAIN)
        return _lib.Metric(self.kind, 1 if dense else 0, self.scalar, p(self.imm), p(self.sqrt_t), p(self.chol_t))

    def _ws_for(self, n_elems):
        nbytes = n_elems * (8 if self.dtype == torch.float64 else 4) + 512
        return self._ws.get(nbytes, self.device)


def gaussian_metric(inverse_mass_matrix, dtype=None, device=None):
    metric = GaussianMetric(inverse_mass_matrix, dtype, device)
    lib = _lib.load()
    code = backend.code(metric.dtype)

    def momentum_generator(srng, num_chains=None, dim=None, transition=None):
        """p[C, d] = M^{1/2} z (metrics.py:65-68).  Shape comes from the metric when it has one."""
        d = metric.dim or dim
        per_chain_kind = metric.kind in (_lib.IMM_DIAG_PER_CHAIN, _lib.IMM_DENSE_PER_CHAIN)
        Cn = num_chains if num_chains is not None else (metric.imm.shape[0] if per_chain_kind else None)
        if d is None or Cn is None:
            raise ValueError("momentum_generator needs num_chains (and dim for a scalar metric)")
        p = torch.empty((Cn, d), dtype=metric.dtype, device=metric.device)
        rng, keep = srng.struct()
        t = srng.transition if transition is None else transition
        rng.transition_offset = 0                  # the transition is passed explicitly
        ws = metric._ws_for(Cn * d)
        m = metric.struct()
        _lib.check(lib.b2h_sample_momentum(backend.context(metric.device), C.byref(m), C.byref(rng), code,
                                           backend.ptr(p), C.c_int64(Cn), C.c_int64(d), C.c_int64(t),
                                           backend.ptr(ws), C.c_int64(ws.numel())))
        return p

    def kinetic_energy(momentum):
        """K[C] = 0.5 p^T imm p (metrics.py:70-73)."""
        p = backend.as_device(momentum, metric.dtype, metric.device)
        Cn, d = p.shape
        K = torch.empty(Cn, dtype=metric.dtype, device=metric.device)
        ws = metric._ws_for(Cn * d)
        m = metric.struct()
        _lib.check(lib.b2h_kinetic_energy(backend.context(metric.device), C.byref(m), code, backend.ptr(p),
                                          backend.ptr(K), C.c_int64(Cn), C.c_int64(d), backend.ptr(ws),
                                          C.c_int64(ws.numel())))
        return K

    def is_turning(momentum_left, momentum_right, momentum_sum):
        """Generalised U-turn criterion (metrics.py:75-104), one bool per chain."""
        pl = backend.as_device(momentum_left, metric.dtype, metric.device)
        pr = backend.as_device(momentum_right, metric.dtype, metric.device)
        ps = backend.as_device(momentum_sum, metric.dtype, metric.device)
        Cn, d = pl.shape
        out = torch.empty(Cn, dtype=torch.uint8, device=metric.device)
        ws = metric._ws_for(2 * Cn * d)
        m = metric.struct()
        _lib.check(lib.b2h_is_turning(backend.context(metric.device), C.byref(m), code, backend.ptr(pl),
                                      backend.ptr(pr), backend.ptr(ps), backend.ptr(out), C.c_int64(Cn),
                                      C.c_int64(d), backend.ptr(ws), C.c_int64(ws.numel())))
        return out.bool()

    for fn in (momentum_generator, kinetic_energy, is_turning):
        fn.metric = metric
    return momentum_generator, kinetic_energy, is_turning
