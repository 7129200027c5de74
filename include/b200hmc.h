/* b200hmc.h -- C-ABI of libb200hmc.so, the B200-native many-chain HMC/NUTS engine.
 *
 * Drop-in boundary for the trajectory hot path of aesara-devs/aehmc.  The
 * reference is pure Python over Aesara and has no FFI of its own; each entry
 * point below names the reference closure it replaces (file:line relative to
 * the reference tree) and is what an Aesara Op's perform() binds through
 * ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - every function returns 0 on success, <0 on error; b2h_last_error() gives a
 *    thread-local message.
 *  - the caller owns every data buffer and passes raw DEVICE pointers unless a
 *    parameter is documented as host.  The library owns only b2h_ctx handles.
 *  - all work is enqueued on the cudaStream_t given at context creation; no call
 *    synchronises unless documented.
 *  - vectors over chains are [C] ; per-chain vectors are row-major [C x d].
 *  - dtype: B2H_F32 / B2H_F64 is the type of positions, momenta, gradients and
 *    energies.  Proposal weights and sum_log_p_accept are always float64
 *    (reference nuts.py:123-124).  Step sizes, draws and diagnostics are float64.
 */
#ifndef B200HMC_H
#define B200HMC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2H_F32 0
#define B2H_F64 1

#define B2H_OK 0
#define B2H_ERR_ARG -1
#define B2H_ERR_CUDA -2
#define B2H_ERR_UNSUPPORTED -3
#define B2H_ERR_WORKSPACE -4

typedef struct b2h_ctx b2h_ctx;

/* ---- log-density models (the reference's user logprob_fn; built-in targets) ---- */
enum {
    B2H_MODEL_IID_GAUSSIAN = 0,  /* a=mu[d], b=inv_var[d], s0 = additive constant of U            */
    B2H_MODEL_CORR_GAUSSIAN = 1, /* a=mu[d], b=precision[d x d] (symmetric, row-major)             */
    B2H_MODEL_FUNNEL = 2,        /* Neal's funnel, q=(v,x_1..x_{d-1})                              */
    B2H_MODEL_EIGHT_SCHOOLS = 3, /* non-centred; a=y[d-2], b=inv_var[d-2]                          */
    B2H_MODEL_LOGISTIC = 4       /* a=X[n_data x d] row-major, b=y[n_data], c=X^T[d x n_data], s0 = 1/prior_scale^2;
                                    s1 = gradient path: 0 FMA/DMMA exactness reference, 2 tcgen05 tensor core
                                    (needs x_bf16 = X and xt_bf16 = X^T as bf16, X bf16-representable; one fused
                                    kernel when dim <= 128), 3 = tensor core, two-kernel formulation (any dim),
                                    4 = fused kernel on two fp16 pieces (needs x_f16 = X * 2^x_f16_shift exactly
                                    representable as fp16, dim <= 128)                                          */
    ,
    B2H_MODEL_USER = 5           /* user-written device function compiled by b2h_user_model_create:
                                    a = the b2h_user_model* handle, b = user data [any length], dtype of the call */
};

typedef struct {
    int32_t kind;
    int32_t dim;
    int64_t n_data;
    const void* a; /* device, dtype of the call */
    const void* b; /* device, dtype of the call */
    const void* c; /* device, model specific (logistic: X^T [d x n_data]) */
    double s0;
    double s1;
    const void* x_bf16;  /* device, logistic tensor-core path: X   [n_data x d] as bf16 */
    const void* xt_bf16; /* device, logistic tensor-core path: X^T [d x n_data] as bf16 */
    const void* x_f16;   /* device, logistic fp16 path: X * 2^x_f16_shift [n_data x d] as fp16 (exact) */
    int32_t x_f16_shift;
    int32_t reserved;
    const double* u_lin; /* device, logistic fp16 path: X^T (1/2 - y) [d] in float64: the part of the potential that is
                            linear in beta, sum_n (1/2 - y_n) x_n . beta, is added outside the contraction kernel */
} b2h_model;

/* ---- gaussian metric (reference metrics.py:10-106) ---- */
enum {
    B2H_IMM_SCALAR = 0,         /* 0-d inverse mass matrix, value in .scalar (host)               */
    B2H_IMM_DIAG = 1,           /* imm[d] shared by all chains                                    */
    B2H_IMM_DIAG_PER_CHAIN = 2, /* imm[C x d] (per-chain adaptation)                              */
    B2H_IMM_DENSE = 3,          /* imm[d x d] symmetric, shared; sqrt = mass_matrix_sqrt[d x d]   */
    B2H_IMM_DENSE_PER_CHAIN = 4 /* imm, sqrt_t, chol_t [C x d x d] row-major, chain c's matrix at c * d * d; each
                                   chain's triple follows the B2H_IMM_DENSE conventions below (reserved bit 0 too) */
};

/* Largest d of a B2H_IMM_DENSE_PER_CHAIN metric.  b2h_dense_factor_per_chain keeps a chain's matrix in the shared
 * memory of one CTA as FP64 (d = 128: 128 KB), and the per-chain metric costs 3 d^2 s bytes per chain (s = dtype size)
 * plus d^2 s for the per-chain Welford state of its adaptation: 4096 chains at d = 128 in FP64 take 1.6 GB + 0.5 GB.
 * Larger d (or chains that share one matrix) want the shared B2H_IMM_DENSE kind: window adaptation with pooled = 1. */
#define B2H_DENSE_PER_CHAIN_MAX_DIM 128

typedef struct {
    int32_t kind;
    int32_t reserved;   /* flags.  bit 0 (dense only): sqrt_t and chol_t are the TRIANGULAR factors described below (sqrt_t
                           lower-, chol_t upper-triangular), so the momentum contractions may skip their zero halves; 0: any
                           factors with sqrt_t^T sqrt_t = imm^-1 and chol_t = (imm sqrt_t^T)^T are read in full            */
    double scalar;
    const void* imm;    /* device; dense: symmetric [d x d] */
    const void* sqrt_t; /* device, dense only: TRANSPOSE of mass_matrix_sqrt = solve_triangular(chol(imm), I,
                           lower, trans) (metrics.py:56-58), row-major [d x d]: p_row = z_row . sqrt_t       */
    const void* chol_t; /* device, dense only: TRANSPOSE of L = chol(imm), row-major [d x d].  imm . p = L L^T L^-T z
                           = L z, so the velocity of a fresh momentum is v_row = z_row . chol_t: the sampler draws p0 and
                           imm . p0 of a transition from the same normals in ONE grouped contraction               */
} b2h_metric;

/* ---- random draws: native Philox4x32-10 or injected (validation mode) ---- */
enum { B2H_RNG_PHILOX = 0, B2H_RNG_INJECTED = 1 };

typedef struct {
    int32_t mode;
    int32_t reserved;
    uint64_t seed;
    uint64_t chain_offset;      /* global id of local chain 0 (multi-GPU sharding)               */
    uint64_t transition_offset; /* global index of the first transition of this call (injected mode:
                                   index of its first row within the T injected transitions)           */
    /* injected draws, float64, device; T = n_injected transitions per chain                     */
    int64_t n_injected;
    const double* z;         /* [C][T][d]                 standard normals (momentum)            */
    const double* u_dir;     /* [C][T][max_depth]         direction: go right iff u > 0.5        */
    const double* u_biased;  /* [C][T][max_depth]         biased progressive sampling            */
    const double* u_uniform; /* [C][T][2^max_depth - 1]   uniform progressive sampling, slot =   */
                             /*                           2^k - 1 + (s - 1) for sub-tree step s  */
    const double* u_accept;  /* [C][T]                    HMC accept                             */
} b2h_rng;

/* ---- per-transition outputs (reference trajectory.py:379-384 Diagnostics) ---- */
typedef struct {
    double* acceptance_probability; /* [C] */
    int32_t* num_doublings;         /* [C] (0 for HMC) */
    uint8_t* is_turning;            /* [C] */
    uint8_t* is_diverging;          /* [C] */
    int32_t* n_leapfrog;            /* [C] integrator steps of the transition (extra) */
} b2h_diag;

/* ---- window adaptation (reference window_adaptation.py:119-227), per chain ---- */
typedef struct {
    int32_t enabled;
    int32_t num_steps;
    const uint8_t* stage;       /* device [num_steps] 0 fast / 1 slow (build_schedule)           */
    const uint8_t* window_end;  /* device [num_steps] is_middle_window_end                       */
    double target_acceptance_rate;
    double gamma, t0, kappa;    /* dual averaging (algorithms.py:17-19)                          */
    double initial_step_size;
    /* state, device, caller-owned so that warm-up can be resumed                                */
    int64_t* da_step;           /* [C] */
    double* da_x;               /* [C] iterates */
    double* da_x_avg;           /* [C] */
    double* da_g_avg;           /* [C] */
    double* da_mu;              /* [C] */
    void* wc_mean;              /* [C x d] dtype */
    void* wc_m2;                /* [C x d] dtype */
    int64_t* wc_n;              /* [C] */
    int32_t pooled;             /* 1: the inverse mass matrix is shared and re-estimated by the CALLER from the pooled
                                   statistics of all chains at each window end (b2h_welford_pooled_update): the engine
                                   runs the per-chain dual averaging only and never touches the metric; any metric kind.
                                   The same mode serves a caller that adapts per-chain DENSE matrices itself
                                   (B2H_IMM_DENSE_PER_CHAIN): it folds the stored draws with b2h_welford_update(full = 1)
                                   and refactors with b2h_dense_factor_per_chain at each window end                   */
    int32_t step_offset;        /* schedule index of the call's first transition (a warm-up run in several calls)    */
} b2h_adapt;

/* ---- sampler configuration ---- */
typedef struct {
    int32_t dtype;
    int32_t max_num_expansions;   /* nuts.py:20 default 10 */
    double divergence_threshold;  /* nuts.py:21 / hmc.py:46 default 1000 */
    int32_t num_integration_steps;/* HMC only (hmc.py:81) */
    int32_t group;                /* threads per chain: 0 = auto, else 1,2,4,8,16,32,128,256 */
    int32_t gradient_path;        /* logistic: 0 auto, 1 FFMA exactness reference, 2 tcgen05 tensor core */
    int32_t thin;                 /* draw storage: keep every thin-th transition of the call (0 or 1: all); slot k of
                                     draws / draw_stats holds transition k * thin */
    int32_t exact_doubling;       /* 0 (default): the reference's sub-trees of 2**k + 1 leapfrogs (trajectory.py:276,302,307),
                                     reproduced decision for decision.  1: balanced sub-trees of 2**k leapfrogs, for which
                                     the iterative U-turn / biased progressive sampling leave the target invariant */
    int32_t reserved;
} b2h_cfg;

/* ======================================================================== */
const char* b2h_last_error(void);
int b2h_version(void);

/* device: CUDA ordinal; stream: cudaStream_t (NULL = legacy default stream) */
int b2h_ctx_create(int device, void* stream, b2h_ctx** out);
int b2h_ctx_destroy(b2h_ctx* ctx);
int b2h_ctx_sync(b2h_ctx* ctx); /* cudaStreamSynchronize */

/* Measurement aid (bench.py's roofline of the integrator / U-turn kernel): with the timer enabled, every launch of the
 * tick kernel of b2h_nuts_run's per-tick engine (the kernel that fuses integrators.py:58-73, termination.py:109-187,
 * trajectory.py:195-273,537-608 for one leapfrog of every chain) is bracketed by a pair of CUDA events on the
 * context's stream.  enable = 2 brackets the model-gradient call of every tick instead (hmc.py:33-34 for all chains: the
 * contraction kernels of logistic regression / the correlated Gaussian, timed inside the step).  b2h_tick_timer(ctx,
 * enable) resets the totals; b2h_tick_timer_read synchronises the stream and returns the summed time and the number
 * of bracketed launches since the last reset.  Off (0) by default. */
int b2h_tick_timer(b2h_ctx* ctx, int32_t enable);
int b2h_tick_timer_read(b2h_ctx* ctx, double* total_ms, int64_t* launches);

/* hmc.new_state (reference hmc.py:16-40): U[C] = -logp(q), g[C x d] = dU/dq */
/* User log-density (the reference's arbitrary Python logprob_fn + aesara.grad, hmc.py:33-34): CUDA C++ source
 * that defines
 *     template <typename T> __device__ T potential_and_grad(const T* q, T* g, int d, const T* data);
 * (returns U(q) = -logprob(q), writes dU/dq into g[0..d)).  Compiled with NVRTC for sm_100a on the current device;
 * the handle goes into b2h_model.a of a B2H_MODEL_USER model.  The compile log is in b2h_last_error() on failure. */
typedef struct b2h_user_model b2h_user_model;
int b2h_user_model_create(const char* cuda_source, b2h_user_model** out);
/* Same, but the source defines only the log-density,
 *     template <typename S, typename T> __device__ S log_density(const S* q, int d, const T* data);
 * written with ordinary arithmetic and exp / log / log1p / sqrt / tanh / sin / cos / square / pow(x, T) / softplus; the
 * gradient comes from forward-mode dual numbers S = Dual<T, dim> (the role of aesara.grad; O(dim) per operation,
 * dim <= 64). */
int b2h_user_model_create_ad(const char* cuda_source, int32_t dim, b2h_user_model** out);
/* Same log_density source, differentiated in reverse mode: S = Var<T> holds the value (.v, as in Dual, so a source
 * that branches on q[i].v compiles in both modes) and a node id.  One evaluation records a tape per chain; one reverse
 * sweep over it gives the gradient, at a cost proportional to the number of operations whatever dim is.  U is
 * bit-identical to the forward mode's; the gradient differs only in the order its terms are summed.
 * 1 <= dim <= B2H_USER_REV_MAX_DIM (the inputs are a per-thread array of dim Vars in local memory).
 *
 * The tape lives in the workspace of every call that evaluates the model (b2h_potential_and_grad, b2h_leapfrog, the
 * engine and the tree builders size it through b2h_potential_workspace_bytes).  With N = the tape capacity in nodes
 * per chain, pitch = C rounded up to a multiple of 32 and E = sizeof(T) (8 for B2H_F64, 4 for B2H_F32):
 *     bytes = 256 + 2 * R(N * pitch * 4) + 2 * R(N * pitch * E) + R((dim + N) * pitch * E),   R(x) = x rounded up to 256
 * (two int32 operand ids and two partials per node, adjoints of the inputs and the nodes; 8 + 3E bytes per node).
 * A smaller workspace returns B2H_ERR_WORKSPACE.  Its contents need not be initialised.
 *
 * The capacity starts at 0.  A chain that needs more nodes than the capacity still computes its values but gets
 * U = +inf and g = 0 (the sampler rejects it as a divergence), and the count it needed is recorded on the device:
 * read it with b2h_user_model_tape_needed after each evaluating call to detect this.  The handle must be used with
 * contexts on the device that was current at creation (B2H_ERR_ARG otherwise). */
#define B2H_USER_REV_MAX_DIM 4096
int b2h_user_model_create_rev(const char* cuda_source, int32_t dim, b2h_user_model** out);
/* Sets the tape capacity in nodes per chain, 0 <= nodes <= 2^31 - 1 - dim.  The workspace size depends on it: a
 * workspace sized before the change may be too small afterwards. */
int b2h_user_model_set_tape_nodes(b2h_user_model* model, int64_t nodes);
/* *needed = the largest node count any chain of a reverse-mode handle needed since the previous read (0 if none was
 * evaluated), then resets it.  Copies on the context's stream and synchronises that stream. */
int b2h_user_model_tape_needed(b2h_ctx* ctx, b2h_user_model* model, int64_t* needed);
int b2h_user_model_destroy(b2h_user_model* model);

int b2h_potential_and_grad(b2h_ctx*, const b2h_model*, int dtype, const void* q, void* U, void* g, int64_t C,
                           void* workspace, int64_t workspace_bytes);
int64_t b2h_potential_workspace_bytes(const b2h_model*, int dtype, int64_t C);

/* gaussian_metric(...)[0] momentum_generator (metrics.py:65-68): p[C x d] = M^{1/2} z */
int b2h_sample_momentum(b2h_ctx*, const b2h_metric*, const b2h_rng*, int dtype, void* p, int64_t C, int64_t d,
                        int64_t transition, void* workspace, int64_t workspace_bytes /* dense: C*d elements */);
/* gaussian_metric(...)[1] kinetic_energy (metrics.py:70-73): K[C] = 0.5 p^T imm p */
int b2h_kinetic_energy(b2h_ctx*, const b2h_metric*, int dtype, const void* p, void* K, int64_t C, int64_t d,
                       void* workspace, int64_t workspace_bytes /* dense: C*d elements */);
/* gaussian_metric(...)[2] is_turning (metrics.py:75-104) */
int b2h_is_turning(b2h_ctx*, const b2h_metric*, int dtype, const void* p_left, const void* p_right,
                   const void* p_sum, uint8_t* out, int64_t C, int64_t d, void* workspace,
                   int64_t workspace_bytes /* dense: 2*C*d elements */);

/* integrators.velocity_verlet one_step x n_steps (integrators.py:58-73; trajectory.static_integration
 * trajectory.py:79-105).  In place on q,p,U,g.  step_size[C] float64; direction[C] int8 (+1/-1) or NULL. */
int b2h_leapfrog(b2h_ctx*, const b2h_model*, const b2h_metric*, int dtype, void* q, void* p, void* U, void* g,
                 const double* step_size, const int8_t* direction, int32_t n_steps, int64_t C,
                 void* workspace, int64_t workspace_bytes);

/* termination.iterative_uturn (termination.py:85-187), batched.  ckpts are [C x max x d]. */
int b2h_termination_update(b2h_ctx*, int dtype, void* momentum_ckpts, void* momentum_sum_ckpts, int64_t* idx_min,
                           int64_t* idx_max, const void* momentum_sum, const void* momentum, const int64_t* step,
                           int64_t C, int64_t d, int32_t max_num_doublings);
int b2h_is_iterative_turning(b2h_ctx*, const b2h_metric*, int dtype, const void* momentum_ckpts,
                             const void* momentum_sum_ckpts, const int64_t* idx_min, const int64_t* idx_max,
                             const void* momentum_sum, const void* momentum, uint8_t* out, int64_t C, int64_t d,
                             int32_t max_num_doublings /* diag-family metrics; dense kinds: B2H_ERR_UNSUPPORTED */);
/* termination._find_storage_indices (termination.py:192-235) */
int b2h_find_storage_indices(b2h_ctx*, const int64_t* step, int64_t* idx_min, int64_t* idx_max, int64_t n);

/* hmc.new_kernel(...)(state, step_size, imm, L) (hmc.py:77-124,157-204): n_transitions HMC transitions per
 * chain with L = cfg->num_integration_steps.  Arguments as b2h_nuts_run (adapt may be NULL). */
int b2h_hmc_run(b2h_ctx*, const b2h_model*, const b2h_metric*, const b2h_rng*, const b2h_cfg*,
                const b2h_adapt* adapt, void* q, void* p, void* U, void* g, double* step_size, int64_t C,
                int32_t n_transitions, b2h_diag* diag, void* draws, double* draw_stats, int32_t n_store,
                int64_t* counters, void* workspace, int64_t workspace_bytes);

/* nuts.new_kernel(...)(state, step_size, imm) (nuts.py:56-153 -> trajectory.py:154-374,428-608):
 * runs the chain state machines until every chain has completed n_transitions transitions
 * (max_ticks <= 0), or for exactly max_ticks leapfrog ticks (chains keep going; the state machine is
 * kept in the workspace and continued when resume != 0).  q,U,g in/out [C x d]; p out.
 * step_size[C] in/out (adapted when adapt.enabled); imm may be DIAG_PER_CHAIN and adapted in place.
 * diag: values of each chain's LAST completed transition.  draws (optional): [n_store][C][d] positions
 * after each of the first n_store transitions; draw_stats (optional) [n_store][C][4] float64 rows of
 * (acceptance_probability, num_doublings, n_leapfrog, flags: bit0 turning, bit1 diverging, bit2 last sub-tree
 * stopped on the iterative U-turn criterion).
 * counters (optional, device int64[4]): total leapfrogs, total transitions, ticks run, active chain-ticks. */
int b2h_nuts_run(b2h_ctx*, const b2h_model*, const b2h_metric*, const b2h_rng*, const b2h_cfg*,
                 const b2h_adapt* adapt, void* q, void* p, void* U, void* g, double* step_size, int64_t C,
                 int32_t n_transitions, int64_t max_ticks, int32_t resume, b2h_diag* diag, void* draws,
                 double* draw_stats, int32_t n_store, int64_t* counters, void* workspace, int64_t workspace_bytes);
int64_t b2h_nuts_workspace_bytes(const b2h_model*, const b2h_metric*, const b2h_cfg*, int64_t C);
/* Threads per chain (1, 8, 32 or 256) a run with cfg->group == 0 will use; free_running != 0: a max_ticks run.  The
 * workspace layout depends on it: a resumed call must run with the group of the call that started the run (pass it
 * as cfg->group). */
int32_t b2h_nuts_plan_group(const b2h_model*, const b2h_metric*, const b2h_cfg*, int64_t C, int32_t free_running);
int64_t b2h_hmc_workspace_bytes(const b2h_model*, const b2h_metric*, const b2h_cfg*, int64_t C);

/* ---- stand-alone trajectory builders with caller-supplied tree state (every model; scalar / diagonal metrics: the
 *      reference's tree state carries no velocities, which the dense-metric engine needs -- use b2h_nuts_run; both
 *      dense kinds return B2H_ERR_UNSUPPORTED) ---- */
typedef struct {
    void *q, *p, *g; /* [C x d] */
    void* U;         /* [C]     */
} b2h_state;

/* trajectory.multiplicative_expansion(...).expand(proposal, left_state, right_state, momentum_sum,
 * termination_state, initial_energy, step_size) (trajectory.py:428-712): all members in/out. */
typedef struct {
    b2h_state proposal;          /* ProposalState.state                                   */
    void* proposal_energy;       /* [C] dtype                                             */
    double* proposal_weight;     /* [C] float64                                           */
    double* proposal_slpa;       /* [C] float64 sum_log_p_accept                          */
    b2h_state left, right;       /* trajectory edges                                      */
    void* momentum_sum;          /* [C x d]                                               */
    void* momentum_ckpts;        /* [C x max_num_expansions x d] TerminationState         */
    void* momentum_sum_ckpts;    /* [C x max_num_expansions x d]                          */
    int64_t *idx_min, *idx_max;  /* [C]                                                   */
    const void* initial_energy;  /* [C] dtype                                             */
} b2h_tree;
int b2h_nuts_expand(b2h_ctx*, const b2h_model*, const b2h_metric*, const b2h_rng*, const b2h_cfg*, b2h_tree* tree,
                    const double* step_size, int64_t C, b2h_diag* diag, void* workspace, int64_t workspace_bytes);

/* trajectory.dynamic_integration(...).integrate(previous_last_state, direction, termination_state, max_num_steps,
 * step_size, initial_energy) (trajectory.py:154-374): one sub-tree of 1 + max_num_steps leapfrogs at most. */
typedef struct {
    b2h_state state;             /* in: previous_last_state; out: last state of the sub-tree */
    const int8_t* direction;     /* [C] +1 / -1                                              */
    b2h_state proposal;          /* out: sub-tree proposal                                   */
    void* proposal_energy;       /* out [C] dtype                                            */
    double* proposal_weight;     /* out [C]                                                  */
    double* proposal_slpa;       /* out [C]                                                  */
    void* momentum_sum;          /* out [C x d] sum of the sub-tree's momenta                */
    void* momentum_ckpts;        /* in/out [C x max_num_expansions x d]                      */
    void* momentum_sum_ckpts;    /* in/out                                                   */
    int64_t *idx_min, *idx_max;  /* in/out [C]                                               */
    const void* initial_energy;  /* [C] dtype                                                */
    int32_t max_num_steps;       /* scan length after the first step (2**k in NUTS)          */
    int32_t expansion;           /* k: selects the uniform-draw slots 2**k - 1 + (s - 1)     */
    int32_t* trajectory_length;  /* out [C]                                                  */
    uint8_t* is_diverging;       /* out [C]                                                  */
    uint8_t* has_terminated;     /* out [C]                                                  */
} b2h_subtree;
int b2h_nuts_subtree(b2h_ctx*, const b2h_model*, const b2h_metric*, const b2h_rng*, const b2h_cfg*, b2h_subtree* sub,
                     const double* step_size, int64_t C, void* workspace, int64_t workspace_bytes);

/* proposals.proposal_generator(...).update scalars (proposals.py:41-52): energy = U + K, delta = E0 - energy
 * (NaN -> -inf), weight = delta, log_p_accept = min(delta, 0), diverging = |delta| > threshold. */
int b2h_proposal_update(b2h_ctx*, int dtype, const void* initial_energy, const void* U, const void* K, double threshold,
                        void* energy, double* weight, double* log_p_accept, uint8_t* is_diverging, int64_t C);
/* proposals.progressive_{uniform,biased}_sampling + maybe_update_proposal scalars (proposals.py:72-174):
 * biased == 0: p = expit(w_new - w_old) (NaN -> 0); biased != 0: p = clip(exp(w_new - w_old), 0, 1).
 * do_accept from the uniform u[C]; weight / sum_log_p_accept merged with logaddexp. */
int b2h_progressive_sampling(b2h_ctx*, int biased, const double* w_old, const double* w_new, const double* slpa_old,
                             const double* slpa_new, const double* u, uint8_t* do_accept, double* w_out,
                             double* slpa_out, int64_t C);
/* row-wise select (maybe_update_proposal / where_proposal): out[c] = mask[c] ? a[c] : b[c], rows of d elements */
int b2h_select_rows(b2h_ctx*, int dtype, const uint8_t* mask, const void* a, const void* b, void* out, int64_t C,
                    int64_t d);

/* hmc.hmc_proposal(...).propose after the static integration (hmc.py:183-204): flips the momentum of the integrated
 * state, delta = (U + K)_old - (U + K)_new (NaN -> -inf), is_diverging = |delta| > threshold, p_accept =
 * clip(exp(delta), 0, 1), Metropolis accept from the uniform u[C] (numpy's binomial(1, p) decision rule).  new_state
 * is overwritten with the final state (the flipped new state, or old_state). */
int b2h_hmc_accept(b2h_ctx*, int dtype, const b2h_state* old_state, b2h_state* new_state, const void* K_old,
                   const void* K_new, const double* u, double threshold, double* p_accept, uint8_t* is_diverging,
                   int64_t C, int64_t d);

/* algorithms.dual_averaging update (algorithms.py:79-115) with gradient = target - p_accept
 * (step_size.py:97); in place on the [C] state arrays. */
int b2h_dual_averaging_update(b2h_ctx*, const double* p_accept, double target, double gamma, double t0, double kappa,
                              int64_t* step, double* x, double* x_avg, double* g_avg, const double* mu, int64_t C);
/* algorithms.welford_covariance update/final (algorithms.py:166-202) and the shrinkage of
 * mass_matrix.covariance_adaptation.final (mass_matrix.py:81-118).  full != 0: m2/out are [C x d x d]. */
int b2h_welford_update(b2h_ctx*, int dtype, const void* value, void* mean, void* m2, int64_t* n, int64_t C,
                       int64_t d, int32_t full);
int b2h_mass_matrix_final(b2h_ctx*, int dtype, const void* m2, const int64_t* n, void* imm_out, int64_t C, int64_t d,
                          int32_t full);

/* Pooled (cross-chain) Welford statistics: the positions of ALL chains in a slow window are one sample of the same
 * target.  Folds a block of draws [T][C][d] into the running float64 state (n, mean[d], m2[d] or, full != 0,
 * m2[d x d]) with the group form of welford_covariance.update (algorithms.py:166-197; Chan's pairwise update), fixed
 * summation order.  n is the number of rows already in the state (host value; the caller adds T * C afterwards). */
int b2h_welford_pooled_update(b2h_ctx*, int dtype, const void* draws, int64_t T, int64_t C, int64_t d, int32_t full,
                              int64_t n, double* mean, double* m2, void* workspace, int64_t workspace_bytes);
int64_t b2h_welford_pooled_workspace_bytes(int64_t T, int64_t C, int64_t d, int32_t full);
/* (n_a, mean_a, m2_a) <- merge with (n_b, mean_b, m2_b): the states of two groups of chains, e.g. two ranks after
 * the all-gather of the adaptation statistics (SURVEY 8e).  scratch_mean: [d] float64. */
int b2h_welford_merge(b2h_ctx*, int64_t d, int32_t full, int64_t n_a, double* mean_a, double* m2_a, int64_t n_b,
                      const double* mean_b, const double* m2_b, double* scratch_mean);

/* Native-RNG draws exported in the injected layout (so a Philox run can be replayed by the oracle). */
int b2h_philox_fill(b2h_ctx*, uint64_t seed, uint64_t chain_offset, uint64_t transition_offset, int64_t C,
                    int64_t n_transitions, int64_t d, int32_t max_depth, double* z, double* u_dir,
                    double* u_biased, double* u_uniform, double* u_accept);

/* Dense apply out[C x d] = in[C x d] . M[d x d] (M symmetric): the mass-matrix / precision mat-vec of all chains */
int b2h_dense_apply(b2h_ctx*, int dtype, const void* in, const void* M, void* out, int64_t C, int64_t d);

/* Per-chain dense apply out[c] = in[c] . M[c] for c < C: in, out [C x d], M [C x d x d] (chain c's matrix at c * d * d),
 * the mat-vec of a B2H_IMM_DENSE_PER_CHAIN metric.  tri: 0 M full, 1 M upper-triangular, 2 M lower-triangular (the
 * codes of b2h_gemm_group.tri; the zero half is never read into a result).  Each element is summed over k in ascending
 * order, so integer inputs give the exact product.  1 <= d <= B2H_DENSE_PER_CHAIN_MAX_DIM. */
int b2h_dense_apply_per_chain(b2h_ctx*, int dtype, const void* in, const void* M, void* out, int64_t C, int64_t d,
                              int32_t tri);
/* Factors the C matrices imm_in [C x d x d] of a B2H_IMM_DENSE_PER_CHAIN metric: imm = (A + A^T) / 2, then in FP64
 * whatever the dtype L = chol(imm), sqrt_t = L^-1 (lower) and chol_t = L^T (upper).  info[c] (device int32 [C]) is 0,
 * or k + 1 when pivot k of chain c is not positive; that chain's imm, sqrt_t and chol_t are then NaN.  imm may alias
 * imm_in.  1 <= d <= B2H_DENSE_PER_CHAIN_MAX_DIM. */
int b2h_dense_factor_per_chain(b2h_ctx*, int dtype, const void* imm_in, void* imm, void* sqrt_t, void* chol_t,
                               int32_t* info, int64_t C, int64_t d);

/* Per-chain mean and unbiased variance (float64 [C x d] each) of draws [T][C][d]: the per-GPU part of R-hat. */
int b2h_chain_moments(b2h_ctx*, int dtype, const void* draws, int64_t T, int64_t C, int64_t d, double* chain_mean,
                      double* chain_var);

/* tcgen05/TMA contraction used by the logistic tensor-core path, exposed for testing:
 * out[z][M x N] (fp32, row pitch ldo, plane stride split_stride) = sum_{p<pieces} A[p*piece_rows + m][k] * B[n][k]
 * with A [pieces*piece_rows x K] and B [N x K] bf16, K contiguous, 16-byte aligned pitches; split-K over z.
 * Plane z sums the k-blocks of 64 [z * kb_per, (z + 1) * kb_per), kb_per = ceil(kb / min(nsplit, kb)) with
 * kb = ceil(K / 64); ceil(kb / kb_per) planes are written.  B2H_ERR_ARG (nothing launched) unless M, N, K, pieces >= 1,
 * piece_rows >= M, lda, ldb >= K, ldo >= N and, when nsplit > 1, split_stride is a multiple of 4 that is at least
 * (M - 1) * ldo + N. */
int b2h_tc_gemm_bf16(b2h_ctx*, const void* A, int64_t lda, const void* B, int64_t ldb, float* out, int64_t M, int64_t N,
                     int64_t K, int32_t pieces, int64_t piece_rows, int64_t ldo, int32_t nsplit, int64_t split_stride);
/* The first product of the two-kernel logistic gradient, exposed for testing: S = sum_p A_p . B^T (as above, one
 * plane) never leaves the SM; the epilogue writes r = sigmoid(S) - y[N] as three bf16 pieces r = p0 + p1 + p2 into R,
 * tile-blocked: piece p, column tile t, row tile u at R + p * r_piece_stride + (t * ceil(M / 128) + u) * 128 * 128,
 * 128 x 128 row-major (columns >= N of rows < M hold 0; rows >= M are not written).  R 1024-byte aligned, y 16-byte
 * aligned.  upart receives the fp64 partial sums of softplus(s) - y s per row: *tiles_per_cta == 0: [column tile][4][M];
 * *tiles_per_cta > 0: [CTA][4][M], CTA b covering the tiles [b, b + 1) * tiles_per_cta of the (row tile, column tile)
 * grid, column tile fastest.  upart must hold 4 * max(ceil(N / 128), SM count) * M doubles. */
int b2h_tc_logistic_residual(b2h_ctx*, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N,
                             int64_t K, int32_t pieces, int64_t piece_rows, const float* y, void* R, int64_t r_piece_stride,
                             double* upart, int32_t* tiles_per_cta);
/* The second product of the two-kernel logistic gradient, exposed for testing: out[z][M x N] = sum_p R_p . B^T (split-K
 * planes as in b2h_tc_gemm_bf16, k-blocks of 64) with R in the tile-blocked layout of b2h_tc_logistic_residual
 * (K = data rows, r_piece_stride >= ceil(K / 128) * ceil(M / 128) * 128 * 128, a multiple of 128), B [N x K] bf16. */
int b2h_tc_gemm_blocked_bf16(b2h_ctx*, const void* R, int64_t r_piece_stride, const void* B, int64_t ldb, float* out,
                             int64_t M, int64_t N, int64_t K, int32_t pieces, int64_t ldo, int32_t nsplit,
                             int64_t split_stride);

/* One problem of a grouped dense contraction (b2h_gemm).  A [M x K] (pitch lda), B [K x N] (pitch ldb) and out
 * (pitch ldo) share the dtype of the call.  m_dev: optional device-side row count (rows r < min(M, *m_dev) are
 * computed).  sub: optional [K] vector subtracted from every row of A.  tri: B is 1 upper- / 2 lower-triangular
 * (the FP64 tensor path then skips the zero k-range of each column tile), 0 general. */
typedef struct {
    const void* A; int64_t lda; const void* B; int64_t ldb; void* out; int64_t ldo;
    int64_t M; const int32_t* m_dev; const void* sub; int32_t tri;
} b2h_gemm_group;

/* The dense contraction behind b2h_dense_apply, the correlated-Gaussian gradient, the momentum contractions of the
 * dense-metric engine and the pooled second moment, exposed for testing: for each of the 1..3 groups,
 * out + s * split_stride (s < nsplit) = the slice-s split-K partial of (A - sub) . B for rows r < min(M, *m_dev). */
int b2h_gemm(b2h_ctx*, int dtype, const b2h_gemm_group* groups, int32_t n_groups, int64_t N, int64_t K, int32_t nsplit,
             int64_t split_stride);

/* Per-chain mean[C x d] and biased autocovariance acov[C x d x (max_lag+1)] (divided by T, the convention of the
 * arviz.ess the reference's tests use, tests/test_hmc.py:158-167) of draws [T][C][d]; building blocks of ESS. */
int b2h_chain_autocov(b2h_ctx*, int dtype, const void* draws, int64_t T, int64_t C, int64_t d, int32_t max_lag,
                      double* mean, double* acov);

#ifdef __cplusplus
}
#endif
#endif /* B200HMC_H */
