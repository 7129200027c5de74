"""ctypes binding of libb200hmc.so (include/b200hmc.h).

There is no CPU fallback: importing a sampler entry point without the built CUDA
library, or creating a context without a B200, raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B2H_LIB: development aid for A/B-ing alternative builds of the same library (still no other implementation)
LIB_PATH = os.environ.get("B2H_LIB") or os.path.join(_HERE, "lib", "libb200hmc.so")

F32, F64 = 0, 1
MODEL_IID_GAUSSIAN, MODEL_CORR_GAUSSIAN, MODEL_FUNNEL, MODEL_EIGHT_SCHOOLS, MODEL_LOGISTIC, MODEL_USER = range(6)
IMM_SCALAR, IMM_DIAG, IMM_DIAG_PER_CHAIN, IMM_DENSE, IMM_DENSE_PER_CHAIN = range(5)
DENSE_PER_CHAIN_MAX_DIM = 128   # B2H_DENSE_PER_CHAIN_MAX_DIM
RNG_PHILOX, RNG_INJECTED = 0, 1


class Model(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("n_data", C.c_int64), ("a", C.c_void_p),
                ("b", C.c_void_p), ("c", C.c_void_p), ("s0", C.c_double), ("s1", C.c_double),
                ("x_bf16", C.c_void_p), ("xt_bf16", C.c_void_p), ("x_f16", C.c_void_p), ("x_f16_shift", C.c_int32),
                ("reserved", C.c_int32), ("u_lin", C.c_void_p)]


class Metric(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("scalar", C.c_double), ("imm", C.c_void_p),
                ("sqrt_t", C.c_void_p), ("chol_t", C.c_void_p)]


class Rng(C.Structure):
    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("seed", C.c_uint64),
                ("chain_offset", C.c_uint64), ("transition_offset", C.c_uint64), ("n_injected", C.c_int64),
                ("z", C.c_void_p), ("u_dir", C.c_void_p), ("u_biased", C.c_void_p), ("u_uniform", C.c_void_p),
                ("u_accept", C.c_void_p)]


class Diag(C.Structure):
    _fields_ = [("acceptance_probability", C.c_void_p), ("num_doublings", C.c_void_p),
                ("is_turning", C.c_void_p), ("is_diverging", C.c_void_p), ("n_leapfrog", C.c_void_p)]


class Adapt(C.Structure):
    _fields_ = [("enabled", C.c_int32), ("num_steps", C.c_int32), ("stage", C.c_void_p),
                ("window_end", C.c_void_p), ("target_acceptance_rate", C.c_double), ("gamma", C.c_double),
                ("t0", C.c_double), ("kappa", C.c_double), ("initial_step_size", C.c_double),
                ("da_step", C.c_void_p), ("da_x", C.c_void_p), ("da_x_avg", C.c_void_p),
                ("da_g_avg", C.c_void_p), ("da_mu", C.c_void_p), ("wc_mean", C.c_void_p),
                ("wc_m2", C.c_void_p), ("wc_n", C.c_void_p), ("pooled", C.c_int32), ("step_offset", C.c_int32)]


class State(C.Structure):
    _fields_ = [("q", C.c_void_p), ("p", C.c_void_p), ("g", C.c_void_p), ("U", C.c_void_p)]


class Tree(C.Structure):
    _fields_ = [("proposal", State), ("proposal_energy", C.c_void_p), ("proposal_weight", C.c_void_p),
                ("proposal_slpa", C.c_void_p), ("left", State), ("right", State), ("momentum_sum", C.c_void_p),
                ("momentum_ckpts", C.c_void_p), ("momentum_sum_ckpts", C.c_void_p), ("idx_min", C.c_void_p),
                ("idx_max", C.c_void_p), ("initial_energy", C.c_void_p)]


class Subtree(C.Structure):
    _fields_ = [("state", State), ("direction", C.c_void_p), ("proposal", State), ("proposal_energy", C.c_void_p),
                ("proposal_weight", C.c_void_p), ("proposal_slpa", C.c_void_p), ("momentum_sum", C.c_void_p),
                ("momentum_ckpts", C.c_void_p), ("momentum_sum_ckpts", C.c_void_p), ("idx_min", C.c_void_p),
                ("idx_max", C.c_void_p), ("initial_energy", C.c_void_p), ("max_num_steps", C.c_int32),
                ("expansion", C.c_int32), ("trajectory_length", C.c_void_p), ("is_diverging", C.c_void_p),
                ("has_terminated", C.c_void_p)]


class Cfg(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("max_num_expansions", C.c_int32), ("divergence_threshold", C.c_double),
                ("num_integration_steps", C.c_int32), ("group", C.c_int32), ("gradient_path", C.c_int32),
                ("thin", C.c_int32), ("exact_doubling", C.c_int32), ("reserved", C.c_int32)]


class GemmGroup(C.Structure):
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int64), ("B", C.c_void_p), ("ldb", C.c_int64), ("out", C.c_void_p),
                ("ldo", C.c_int64), ("M", C.c_int64), ("m_dev", C.c_void_p), ("sub", C.c_void_p), ("tri", C.c_int32)]


# every symbol include/b200hmc.h declares (tests check the .so exports all of them)
EXPORTS = [
    "b2h_last_error", "b2h_version", "b2h_ctx_create", "b2h_ctx_destroy", "b2h_ctx_sync",
    "b2h_potential_and_grad", "b2h_potential_workspace_bytes", "b2h_sample_momentum", "b2h_kinetic_energy",
    "b2h_is_turning", "b2h_leapfrog", "b2h_termination_update", "b2h_is_iterative_turning",
    "b2h_find_storage_indices", "b2h_hmc_run", "b2h_nuts_run", "b2h_nuts_workspace_bytes",
    "b2h_hmc_workspace_bytes", "b2h_dual_averaging_update", "b2h_welford_update", "b2h_mass_matrix_final",
    "b2h_philox_fill", "b2h_dense_apply", "b2h_dense_apply_per_chain", "b2h_dense_factor_per_chain", "b2h_chain_moments", "b2h_chain_autocov", "b2h_tc_gemm_bf16", "b2h_tc_logistic_residual",
    "b2h_tc_gemm_blocked_bf16", "b2h_gemm", "b2h_nuts_expand", "b2h_nuts_subtree", "b2h_proposal_update",
    "b2h_progressive_sampling", "b2h_select_rows", "b2h_user_model_create", "b2h_user_model_create_ad", "b2h_user_model_create_rev",
    "b2h_user_model_create_warp",
    "b2h_user_model_set_tape_nodes", "b2h_user_model_tape_needed", "b2h_user_model_destroy",
    "b2h_hmc_accept", "b2h_nuts_plan_group", "b2h_welford_pooled_update", "b2h_welford_pooled_workspace_bytes", "b2h_welford_merge",
    "b2h_tick_timer", "b2h_tick_timer_read",
]

_lib = None


class B200HMCError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it was not built: the package never
    falls back to another implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200HMCError(
            f"{LIB_PATH} not found: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "aehmc_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.b2h_last_error.restype = C.c_char_p
    for name in ("b2h_potential_workspace_bytes", "b2h_nuts_workspace_bytes", "b2h_hmc_workspace_bytes",
                 "b2h_welford_pooled_workspace_bytes"):
        getattr(lib, name).restype = C.c_int64
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise B200HMCError(f"libb200hmc error {rc}: {load().b2h_last_error().decode()}")
