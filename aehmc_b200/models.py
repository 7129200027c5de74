"""Built-in log-density models: the ``logprob_fn`` argument of hmc/nuts.new_kernel.

The reference takes an arbitrary Python ``logprob_fn`` and differentiates it with
aesara.grad (reference hmc.py:33-34).  The CUDA engine needs the gradient as device
code, so ``logprob_fn`` is a model descriptor here; calling it returns the log-density
like the reference's function would.  Definitions match oracle/models.py.
"""
from __future__ import annotations

import ctypes as C

import math

import numpy as np
import torch

from . import _lib, backend

EIGHT_SCHOOLS_Y = (28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0)
EIGHT_SCHOOLS_SIGMA = (15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0)


class Model:
    kind = -1
    dim = 0

    def __init__(self, dtype=torch.float64, device=None):
        self.dtype = backend.torch_dtype(dtype)
        self.device = backend.device(device)
        self._ws = backend.Workspace()

    # -- C-ABI view ---------------------------------------------------------------------------
    def struct(self):
        raise NotImplementedError

    # -- hmc.new_state (reference hmc.py:16-40) ----------------------------------------------------
    def potential_and_grad(self, q):
        """U[C], dU/dq[C,d] for positions q[C,d]."""
        U, g = self._evaluate(q)
        self.check_tape()
        return U, g

    def check_tape(self):
        """Raise if a chain evaluated since the last check needed more tape than a reverse-mode user model holds (its
        U was +inf and its gradient 0).  Called after every call that evaluates the model; a no-op for every other
        model."""

    def _evaluate(self, q):
        q = backend.as_device(q, self.dtype, self.device)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"position must be [chains, {self.dim}], got {tuple(q.shape)}")
        lib = _lib.load()
        Cn = q.shape[0]
        U = torch.empty(Cn, dtype=self.dtype, device=self.device)
        g = torch.empty_like(q)
        m = self.struct()
        nbytes = lib.b2h_potential_workspace_bytes(C.byref(m), backend.code(self.dtype), C.c_int64(Cn))
        ws = self._ws.get(nbytes, self.device)
        _lib.check(lib.b2h_potential_and_grad(backend.context(self.device), C.byref(m), backend.code(self.dtype),
                                              backend.ptr(q), backend.ptr(U), backend.ptr(g), C.c_int64(Cn),
                                              backend.ptr(ws), C.c_int64(ws.numel())))
        return U, g

    def __call__(self, q):
        """log-density, like the reference's ``logprob_fn(q)``."""
        return -self.potential_and_grad(q)[0]


class IIDGaussian(Model):
    kind = _lib.MODEL_IID_GAUSSIAN

    def __init__(self, mu, sigma, const=0.0, dtype=torch.float64, device=None):
        super().__init__(dtype, device)
        sigma = np.asarray(sigma, dtype=np.float64)
        self.mu = backend.as_device(np.asarray(mu, dtype=np.float64), self.dtype, self.device)
        self.inv_var = backend.as_device(1.0 / (sigma * sigma), self.dtype, self.device)
        self.const = float(const)
        self.dim = int(self.mu.numel())

    def struct(self):
        return _lib.Model(self.kind, self.dim, 0, self.mu.data_ptr(), self.inv_var.data_ptr(), None, self.const, 0.0,
                          None, None)


class CorrelatedGaussian(Model):
    kind = _lib.MODEL_CORR_GAUSSIAN

    def __init__(self, mu, precision, dtype=torch.float64, device=None):
        super().__init__(dtype, device)
        self.mu = backend.as_device(np.asarray(mu, dtype=np.float64), self.dtype, self.device)
        prec = np.asarray(precision.cpu() if isinstance(precision, torch.Tensor) else precision, dtype=np.float64)
        self.precision = backend.as_device(0.5 * (prec + prec.T), self.dtype, self.device)
        self.dim = int(self.mu.numel())

    def struct(self):
        return _lib.Model(self.kind, self.dim, 0, self.mu.data_ptr(), self.precision.data_ptr(), None, 0.0, 0.0,
                          None, None)


class NealFunnel(Model):
    kind = _lib.MODEL_FUNNEL

    def __init__(self, dim=10, dtype=torch.float64, device=None):
        super().__init__(dtype, device)
        self.dim = int(dim)

    def struct(self):
        return _lib.Model(self.kind, self.dim, 0, None, None, None, 0.0, 0.0, None, None)


class EightSchools(Model):
    kind = _lib.MODEL_EIGHT_SCHOOLS

    def __init__(self, y=EIGHT_SCHOOLS_Y, sigma=EIGHT_SCHOOLS_SIGMA, dtype=torch.float64, device=None):
        super().__init__(dtype, device)
        sigma = np.asarray(sigma, dtype=np.float64)
        self.y = backend.as_device(np.asarray(y, dtype=np.float64), self.dtype, self.device)
        self.inv_var = backend.as_device(1.0 / (sigma * sigma), self.dtype, self.device)
        self.dim = 2 + int(self.y.numel())

    def struct(self):
        return _lib.Model(self.kind, self.dim, 0, self.y.data_ptr(), self.inv_var.data_ptr(), None, 0.0, 0.0,
                          None, None)


class LogisticRegression(Model):
    """``tensor_core=True`` evaluates the batched gradient X.B / X^T.R on tcgen05 tensor cores (bf16 operands,
    beta and the residuals split into three bf16 pieces, fp32 accumulation in TMEM): fp32-class accuracy.  It
    needs X to be bf16-representable.  With dim <= 128 the two products and the residual run as ONE kernel (S in
    TMEM, residual pieces written back to TMEM as the A operand of the second product).  When, in addition,
    X * 2^k is exactly representable in fp16 for some k (true for bf16 data spanning less than 2^32 in magnitude),
    beta and the residual are carried as TWO fp16 pieces (22 significant bits) with beta resident in TMEM: two
    thirds of the tensor work.  ``tensor_core="bf16x3"`` forces the three-piece bf16 kernel,
    ``tensor_core="two_kernel"`` the formulation that passes the residual pieces through memory (any dim).
    Real-valued features are not bf16-representable: ``round_features=True`` rounds X to bf16 once, up front, so that
    the model itself is defined on the rounded features (a relative perturbation of at most 2^-9 per entry).
    The default (``False``) is the FP64/FP32 FMA-DMMA path (exactness reference)."""
    kind = _lib.MODEL_LOGISTIC

    def __init__(self, X, y, prior_scale=1.0, dtype=torch.float64, device=None, tensor_core=False, round_features=False):
        super().__init__(dtype, device)
        self.X = backend.as_device(X, self.dtype, self.device)
        if round_features:
            # the MODEL becomes the one with bf16-rounded features (every gradient path then sees the same X)
            self.X = self.X.to(torch.bfloat16).to(self.dtype)
        self.Xt = self.X.t().contiguous()
        self.y = backend.as_device(y, self.dtype, self.device)
        self.inv_prior_var = 1.0 / float(prior_scale) ** 2
        self.n_data, self.dim = int(self.X.shape[0]), int(self.X.shape[1])
        self.tensor_core = bool(tensor_core)
        self.tc_flag = 3.0 if tensor_core == "two_kernel" else (2.0 if self.tensor_core else 0.0)
        self.X_bf16 = self.Xt_bf16 = self.X_f16 = self.u_lin = None
        self.x_f16_shift = 0
        if self.tensor_core:
            xb = self.X.to(torch.bfloat16)
            if not torch.equal(xb.to(self.dtype), self.X):
                raise ValueError("tensor_core=True needs a bf16-representable design matrix X")
            if self.n_data % 8 or self.dim % 8:
                raise ValueError("tensor_core=True needs n_data and dim to be multiples of 8 (16-byte TMA pitches)")
            self.X_bf16 = xb.contiguous()
            self.Xt_bf16 = xb.t().contiguous()
            if tensor_core is True and self.dim <= 128:
                # fp16 copy X * 2^shift (exact): largest magnitude just below 2^15
                amax = float(self.X.abs().max())
                if amax > 0.0 and math.isfinite(amax):
                    shift = 14 - int(math.floor(math.log2(amax)))
                    xs = torch.ldexp(self.X.double(), torch.tensor(shift, device=self.device))
                    xh = xs.to(torch.float16)
                    if bool(torch.isfinite(xh).all()) and torch.equal(xh.double(), xs):
                        self.X_f16, self.x_f16_shift, self.tc_flag = xh.contiguous(), shift, 4.0
                        # sum_n (1/2 - y_n) x_n: the potential's part that is linear in beta
                        self.u_lin = (self.X.double().t() @ (0.5 - self.y.double())).contiguous()

    def struct(self):
        p = lambda t: None if t is None else t.data_ptr()
        return _lib.Model(self.kind, self.dim, self.n_data, self.X.data_ptr(), self.y.data_ptr(),
                          self.Xt.data_ptr(), self.inv_prior_var, self.tc_flag,
                          p(self.X_bf16), p(self.Xt_bf16), p(self.X_f16), self.x_f16_shift, 0, p(self.u_lin))


class UserModel(Model):
    """A log-density written by the user as CUDA C++ (the reference's arbitrary ``logprob_fn``; SURVEY 8f row 3).

    ``source`` must define::

        template <typename T>
        __device__ T potential_and_grad(const T* q, T* g, int d, const T* data);   // returns U = -logprob, writes dU/dq

    or, with ``autodiff=True``, only the log-density::

        template <typename S, typename T>
        __device__ S log_density(const S* q, int d, const T* data);                 // returns logprob

    written with ordinary arithmetic and exp / log / log1p / sqrt / tanh / sin / cos / square / pow / softplus: the
    gradient then comes from automatic differentiation (the role of ``aesara.grad``).  Up to dim 64 it is forward mode,
    dual numbers carrying all dim partials (O(dim) per operation); above, reverse mode: each chain records a tape of
    its operations in the workspace and one reverse sweep gives the gradient (O(1) per operation, dim <= 4096).  The
    tape capacity is probed once here, by evaluating q = 0; a density whose operation count depends on q must pass
    ``tape_nodes`` (nodes per chain) instead.  A chain that needs more raises ``B200HMCError`` after the call that
    evaluated it.  It is compiled once with NVRTC for sm_100a (``b2h_user_model_create[_ad|_rev]``) and evaluated one
    thread per chain;
    the sampler runs it in split mode (one gradient launch per leapfrog tick).  ``data`` is an optional flat array of
    constants handed to the function in the model's dtype.  ``host_fn(q[d]) -> (U, g)`` is an optional NumPy
    counterpart (used by the tests as the oracle's model); it is never called by the sampler.

    ``warp=True`` declares that the source is written in the warp calling convention
    (``b2h_user_model_create_warp``): each chain is evaluated by one full warp, and the function takes one more
    argument, ``const Warp& w``::

        template <typename T>
        __device__ T potential_and_grad(const T* q, T* g, int d, const T* data, const Warp& w);
        template <typename S, typename T>                                           // autodiff=True
        __device__ S log_density(const S* q, int d, const T* data, const Warp& w);

    All 32 lanes call it; the typical loop is ``for (int i = w.lane; i < d; i += w.size)``.  ``w.sum(x)`` (for T and
    S) returns the sum over the lanes, bit-identical on every lane; every lane must call each ``w.sum`` in the same
    order, and calling it from lane-divergent code is undefined.  U is lane 0's return value (with autodiff, the
    gradient is that of lane 0's value), so the other lanes' contributions must reach lane 0 through ``w.sum``.  In
    the hand-written form each element of g is written by exactly one lane.  With autodiff the warp form is reverse
    mode at every dim (each lane records its own tape; ``tape_nodes`` counts nodes per lane) and its gradient is
    deterministic.  It suits wide models: the chain's work is spread over 32 lanes."""
    kind = _lib.MODEL_USER
    FORWARD_MAX_DIM = 64          # autodiff: forward mode up to this dim, reverse mode above

    def __init__(self, source, dim, data=None, dtype=torch.float64, device=None, host_fn=None, autodiff=False,
                 tape_nodes=None, warp=False):
        super().__init__(dtype, device)
        self.dim = int(dim)
        self.autodiff = bool(autodiff)
        self.warp = bool(warp)
        self.reverse = self.autodiff and (self.warp or self.dim > self.FORWARD_MAX_DIM)
        if tape_nodes is not None and not self.reverse:
            raise ValueError(f"tape_nodes applies to reverse-mode models (autodiff=True, dim > {self.FORWARD_MAX_DIM}, "
                             "or warp=True)")
        self.tape_nodes = 0
        self.source = str(source)
        self.host_fn = host_fn
        self.data = None if data is None else backend.as_device(np.asarray(data, dtype=np.float64).ravel(), self.dtype,
                                                                self.device)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            handle = C.c_void_p()
            if self.warp:
                _lib.check(lib.b2h_user_model_create_warp(self.source.encode(), C.c_int32(self.dim),
                                                          C.c_int32(int(self.autodiff)), C.byref(handle)))
            elif self.reverse:
                _lib.check(lib.b2h_user_model_create_rev(self.source.encode(), C.c_int32(self.dim), C.byref(handle)))
            elif self.autodiff:
                _lib.check(lib.b2h_user_model_create_ad(self.source.encode(), C.c_int32(self.dim), C.byref(handle)))
            else:
                _lib.check(lib.b2h_user_model_create(self.source.encode(), C.byref(handle)))
        self._handle = handle
        self._lib = lib
        if self.reverse:
            if tape_nodes is None:
                self._evaluate(torch.zeros((1, self.dim), dtype=self.dtype, device=self.device))
                tape_nodes = self._tape_needed()
            _lib.check(lib.b2h_user_model_set_tape_nodes(handle, C.c_int64(int(tape_nodes))))
            self.tape_nodes = int(tape_nodes)

    def _tape_needed(self):
        n = C.c_int64()
        _lib.check(self._lib.b2h_user_model_tape_needed(backend.context(self.device), self._handle, C.byref(n)))
        return n.value

    def check_tape(self):
        if self.reverse:
            n = self._tape_needed()
            if n > self.tape_nodes:
                per = "a lane of a chain" if self.warp else "a chain"
                raise _lib.B200HMCError(f"reverse-mode user model: {per} needed {n} tape nodes, the capacity is "
                                        f"{self.tape_nodes} (pass tape_nodes >= {n} to UserModel)")

    def struct(self):
        return _lib.Model(self.kind, self.dim, 0, self._handle.value, None if self.data is None else self.data.data_ptr(),
                          None, 0.0, 0.0, None, None)

    def __del__(self):
        h, self._handle = getattr(self, "_handle", None), None
        if h is not None and h.value:
            try:
                self._lib.b2h_user_model_destroy(h)
            except Exception:
                pass
