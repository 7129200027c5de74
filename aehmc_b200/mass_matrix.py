"""covariance_adaptation (reference mass_matrix.py:12-120) over batched chains."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib, algorithms, backend


def covariance_adaptation(is_mass_matrix_full=False):
    wc_init, wc_update, wc_final = algorithms.welford_covariance(is_mass_matrix_full)
    lib = _lib.load()
    full = 1 if is_mass_matrix_full else 0

    def init(n_dims, num_chains=1, dtype=torch.float64, device=None):
        dev = backend.device(device)
        if is_mass_matrix_full:
            imm = torch.eye(n_dims, dtype=dtype, device=dev).expand(num_chains, n_dims, n_dims).contiguous()
        else:
            imm = torch.ones((num_chains, n_dims), dtype=dtype, device=dev)
        return imm, wc_init(n_dims, num_chains, dtype, dev)

    def update(position, wc_state):
        return wc_update(position, *wc_state)

    def final(wc_state):
        """Stan's shrinkage (mass_matrix.py:103-116): (n/(n+5)) cov + 1e-3 (5/(n+5)) [* I]."""
        _, m2, n = wc_state
        out = torch.empty_like(m2)
        Cn, d = m2.shape[0], m2.shape[1]
        _lib.check(lib.b2h_mass_matrix_final(backend.context(m2.device), backend.code(m2.dtype), backend.ptr(m2),
                                             backend.ptr(n), backend.ptr(out), C.c_int64(Cn), C.c_int64(d),
                                             C.c_int32(full)))
        return out

    return init, update, final


def merge_welford(n_a, mean_a, m2_a, n_b, mean_b, m2_b):
    """Chan's pairwise merge of two Welford states (the group form of algorithms.py:187-197), float64, on whatever
    device the tensors live: the reduction operator of the cross-rank adaptation exchange."""
    if n_b == 0:
        return n_a, mean_a, m2_a
    if n_a == 0:
        return n_b, mean_b.clone(), m2_b.clone()
    n = n_a + n_b
    delta = mean_b - mean_a
    cross = torch.outer(delta, delta) if m2_a.ndim == 2 else delta * delta
    return n, mean_a + delta * (n_b / n), m2_a + m2_b + cross * (n_a * n_b / n)


class PooledWelford:
    """Cross-chain Welford state of one slow window: (n, mean[d], m2[d] or m2[d, d]) in float64 over the positions of
    ALL chains (and, after ``all_reduce``, all ranks).  ``update`` folds a block of draws [T, C, d] on the device
    (``b2h_welford_pooled_update``); ``all_reduce`` all-gathers the per-rank states (NCCL over NVLink on GPUs, gloo in
    the CPU tests) and merges them in rank order, so every rank ends with the same bits; ``final`` applies the
    reference's shrinkage (mass_matrix.py:103-116)."""

    def __init__(self, n_dims, is_mass_matrix_full=False, device=None):
        self.d, self.full = int(n_dims), bool(is_mass_matrix_full)
        self.device = torch.device(device) if device is not None else backend.device(None)
        self._ws = backend.Workspace()
        self.reset()

    def reset(self):
        self.n = 0
        self.mean = torch.zeros(self.d, dtype=torch.float64, device=self.device)
        self.m2 = torch.zeros((self.d, self.d) if self.full else (self.d,), dtype=torch.float64, device=self.device)

    def update(self, draws):
        """draws [T, C, d] (or [C, d]) CUDA tensor, float32 or float64."""
        x = draws if draws.ndim == 3 else draws.unsqueeze(0)
        x = x.contiguous()
        T, Cn, d = x.shape
        if d != self.d:
            raise ValueError("draws and state dimensions differ")
        lib = _lib.load()
        full = C.c_int32(1 if self.full else 0)
        nbytes = lib.b2h_welford_pooled_workspace_bytes(C.c_int64(T), C.c_int64(Cn), C.c_int64(d), full)
        ws = self._ws.get(nbytes, x.device)
        _lib.check(lib.b2h_welford_pooled_update(backend.context(x.device), backend.code(x.dtype), backend.ptr(x),
                                                 C.c_int64(T), C.c_int64(Cn), C.c_int64(d), full, C.c_int64(self.n),
                                                 backend.ptr(self.mean), backend.ptr(self.m2), backend.ptr(ws),
                                                 C.c_int64(ws.numel())))
        self.n += T * Cn

    def all_reduce(self):
        """Merge the states of all ranks (no-op without an initialised process group)."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return self
        world = dist.get_world_size()
        flat = torch.cat([torch.tensor([float(self.n)], dtype=torch.float64, device=self.device), self.mean,
                          self.m2.reshape(-1)])
        parts = [torch.empty_like(flat) for _ in range(world)]
        dist.all_gather(parts, flat)
        n, mean, m2 = 0, torch.zeros_like(self.mean), torch.zeros_like(self.m2)
        for part in parts:                                  # fixed (rank) order: identical bits on every rank
            n, mean, m2 = merge_welford(n, mean, m2, int(round(float(part[0]))), part[1:1 + self.d],
                                        part[1 + self.d:].reshape(self.m2.shape))
        self.n, self.mean, self.m2 = n, mean.contiguous(), m2.contiguous()
        return self

    def final(self, dtype=torch.float64):
        """inverse mass matrix [d] or [d, d]: (n/(n+5)) m2/(n-1) + 1e-3 (5/(n+5)) [* I] (mass_matrix.py:103-116)."""
        n = float(self.n)
        cov = self.m2 / (n - 1.0)
        scaled = (n / (n + 5.0)) * cov
        shrink = 1e-3 * (5.0 / (n + 5.0))
        out = scaled + shrink * torch.eye(self.d, dtype=torch.float64, device=self.device) if self.full else scaled + shrink
        return out.to(dtype)


class PerChainWelford:
    """Per-chain Welford state of one slow window for dense per-chain adaptation: (mean [C, d], m2 [C, d, d], n [C])
    in the dtype of the draws, the state of the reference's welford_covariance run once per chain.  ``update`` folds a
    block of draws [T, C, d] one transition at a time, in order, with the reference's recurrence
    (``b2h_welford_update``, algorithms.py:166-197, in place); ``final`` applies the shrinkage of
    mass_matrix.py:103-116 and returns imm [C, d, d]."""

    def __init__(self, num_chains, n_dims, dtype, device):
        self.C, self.d, self.dtype, self.device = int(num_chains), int(n_dims), dtype, device
        self.mean = torch.zeros((self.C, self.d), dtype=dtype, device=device)
        self.m2 = torch.zeros((self.C, self.d, self.d), dtype=dtype, device=device)
        self.n = torch.zeros(self.C, dtype=torch.int64, device=device)

    def reset(self):
        self.mean.zero_()
        self.m2.zero_()
        self.n.zero_()

    def update(self, draws):
        x = backend.as_device(draws, self.dtype, self.device)
        lib, ctx, code = _lib.load(), backend.context(self.device), backend.code(self.dtype)
        for t in range(x.shape[0]):
            _lib.check(lib.b2h_welford_update(ctx, code, backend.ptr(x[t]), backend.ptr(self.mean), backend.ptr(self.m2),
                                              backend.ptr(self.n), C.c_int64(self.C), C.c_int64(self.d), C.c_int32(1)))

    def all_reduce(self):
        """Nothing to merge: every chain keeps its own statistics."""
        return self

    def final(self, dtype=None):
        return covariance_adaptation(True)[2]((self.mean, self.m2, self.n))
