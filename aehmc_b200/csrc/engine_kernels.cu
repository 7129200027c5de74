// Kernels and launch logic of the tick engine (see engine.cuh).
//
//  fused mode : model gradient is a device function (iid Gaussian, funnel, eight
//               schools) and the metric is scalar/diagonal -> ONE persistent kernel
//               runs every chain through all its ticks; nothing returns to the host.
//  split mode : gradient and/or metric need an all-chain contraction (dense metric,
//               correlated Gaussian, logistic regression) -> each tick is
//               pre (half kick + drift) -> gradient -> [dense metric: w' = imm.g', one contraction] -> post,
//               all chains in lock-step, chains restarting transitions independently.
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "engine_host.cuh"

namespace b2h {

// ---------------------------------------------------------------------------
// workspace carving
// ---------------------------------------------------------------------------
struct Carver {
    char* base;
    size_t off;
    template <typename U>
    U* take(size_t n) {
        off = (off + 255) & ~(size_t)255;
        U* p = base ? (U*)(base + off) : nullptr;
        off += n * sizeof(U);
        return p;
    }
};

static int auto_group(int d, long long C, int model_kind, bool free_running) {
    // Tiny targets: thread per chain (the whole front in the thread's registers, fused_run_kernel E = 10 / 16) once there
    // are enough chains to fill the machine with threads.  Measured on config 4 (65536 chains, d = 10,
    // benchmarks/c4_tail_probe.py): eight schools 1.01 vs 0.64 G evals/s free-running and 0.70 vs 0.54 for a fixed
    // number of transitions; the funnel's deep trees run better on 8 lanes (free-running 0.79 vs 0.59-0.74), and its
    // per-chain work is so heavy-tailed (max / mean = 16-24) that a fixed number of transitions is bound by the slowest
    // chains, where a lone chain steps faster on 8 lanes (7 vs 11 us per leapfrog).
    if (d <= 16) {
        if (model_kind == B2H_MODEL_FUNNEL) return C >= 262144 ? 1 : 8;
        return C >= 32768 ? 1 : 8;
    }
    if (d <= 64) return 8;
    if (d <= 512) return 32;
    return 256;
}

static bool model_is_fused(int kind) {
    return kind == B2H_MODEL_IID_GAUSSIAN || kind == B2H_MODEL_FUNNEL || kind == B2H_MODEL_EIGHT_SCHOOLS;
}

static int make_plan(const b2h_model* model, const b2h_metric* metric, const b2h_cfg* cfg, EnginePlan& pl,
                     long long C = 0, bool free_running = false) {
    pl.dense_per_chain = metric->kind == B2H_IMM_DENSE_PER_CHAIN;
    pl.dense = metric->kind == B2H_IMM_DENSE || pl.dense_per_chain;
    if (pl.dense_per_chain && (model->dim < 1 || model->dim > B2H_DENSE_PER_CHAIN_MAX_DIM)) {
        set_error("a per-chain dense metric needs 1 <= d <= " + std::to_string(B2H_DENSE_PER_CHAIN_MAX_DIM) +
                  " (B2H_DENSE_PER_CHAIN_MAX_DIM); for larger d adapt one shared dense matrix (pooled=True)");
        return B2H_ERR_ARG;
    }
    pl.per_chain_imm = metric->kind == B2H_IMM_DIAG_PER_CHAIN;
    pl.scalar_imm = metric->kind == B2H_IMM_SCALAR;
    pl.split = pl.dense || !model_is_fused(model->kind);
    int G = cfg->group > 0 ? cfg->group : auto_group(model->dim, C, model->kind, free_running);
    if (pl.split && G < 8) G = 8;          // split scratch is row-major: needs the row-major layout
    if (G != 1 && G != 8 && G != 32 && G != 256) {
        set_error("group must be one of 0 (auto), 1, 8, 32, 256");
        return B2H_ERR_ARG;
    }
    if ((model->kind == B2H_MODEL_FUNNEL || model->kind == B2H_MODEL_EIGHT_SCHOOLS) && !pl.split && G > 8) G = 8;
    pl.G = G;
    return 0;
}

template <typename T>
static size_t carve(EngineView<T>& v, char* base, const EnginePlan& pl, const b2h_model* model, int C, int d,
                    int maxd, bool adapt, size_t model_ws_bytes, size_t* model_ws_off) {
    Carver cv{base, 0};
    const size_t n = (size_t)C * d;
    v.ql = cv.take<T>(n); v.pl = cv.take<T>(n); v.gl = cv.take<T>(n);
    v.qr = cv.take<T>(n); v.pr = cv.take<T>(n); v.gr = cv.take<T>(n);
    v.qs = cv.take<T>(n); v.ps = cv.take<T>(n); v.gs = cv.take<T>(n);
    v.qp = cv.take<T>(n); v.pp = cv.take<T>(n); v.gp = cv.take<T>(n);
    v.msum = cv.take<T>(n); v.sms = cv.take<T>(n);
    v.mck = cv.take<T>(n * maxd); v.sckp = cv.take<T>(n * maxd);
    v.vl = v.vr = v.vck = nullptr;
    v.wl = v.wr = v.ws = v.wp = nullptr;
    if (pl.dense) {
        v.vl = cv.take<T>(n); v.vr = cv.take<T>(n); v.vck = cv.take<T>(n * maxd);
        v.wl = cv.take<T>(n); v.wr = cv.take<T>(n); v.ws = cv.take<T>(n); v.wp = cv.take<T>(n);
    }
    v.rec = cv.take<ChainRec>(C);
    T* imm_own = nullptr;
    if (pl.per_chain_imm) imm_own = cv.take<T>(n);
    else if (pl.scalar_imm) imm_own = cv.take<T>(1);
    v.imm = imm_own;
    v.adapt.wc_mean = v.adapt.wc_m2 = nullptr;
    if (adapt) { v.adapt.wc_mean = cv.take<T>(n); v.adapt.wc_m2 = cv.take<T>(n); }
    v.xa = v.xb = v.xc = v.Unew = nullptr;
    v.u_center = nullptr;
    v.mom_p = v.mom_v = v.mom_z = nullptr; v.mom_count = nullptr; v.mom_list = nullptr;
    if (pl.split) {
        v.xa = cv.take<T>(n); v.xb = cv.take<T>(n); v.Unew = cv.take<T>(C);
    }
    if (pl.dense) {
        v.xc = cv.take<T>(n);
        v.mom_p = cv.take<T>(n); v.mom_v = cv.take<T>(n); v.mom_z = cv.take<T>(2 * n);
        v.mom_count = cv.take<int>(4); v.mom_list = cv.take<int>(2 * (size_t)C);
        // the shared matrix's rider is a split-K contraction; the per-chain one writes its rows directly
        v.mom_part = pl.dense_per_chain ? nullptr : cv.take<T>(2 * (size_t)kRiderSplit * n);
    }
    v.scratch = cv.take<int>(64);
    if (model_ws_bytes) {
        cv.off = (cv.off + 255) & ~(size_t)255;
        if (model_ws_off) *model_ws_off = cv.off;
        cv.off += model_ws_bytes;
    }
    return cv.off + 256;
}

// ---------------------------------------------------------------------------
// entry / exit kernels (user row-major arrays <-> engine layout)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void copy_in_kernel(EngineView<T> v, const T* q, const T* g, const T* U, const double* eps,
                               const T* imm_user, T imm_scalar, int write_scalar, double init_step_size) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0 && write_scalar) v.imm[0] = imm_scalar;
    if (idx >= (i64)v.C * v.d) return;
    int c = (int)(idx / v.d), j = (int)(idx % v.d);
    i64 a = (i64)c * v.sc + (i64)j * v.sj;
    v.qp[a] = q[idx];
    v.gp[a] = g[idx];
    if (imm_user) v.imm[a] = imm_user[idx];
    if (v.adapt.enabled && v.adapt.wc_mean) { ((T*)v.adapt.wc_mean)[a] = 0; ((T*)v.adapt.wc_m2)[a] = 0; }
    if (j == 0) {
        ChainRec r;
        memset(&r, 0, sizeof(r));
        r.phase = PH_START;
        r.U_prop = (double)U[c];
        r.eps = eps[c];
        if (v.adapt.enabled && v.adapt.step_offset == 0) {
            // window_adaptation.init (window_adaptation.py:132-144): mu = initial step size, step size = exp(0)
            v.adapt.da_step[c] = 1; v.adapt.da_x[c] = 0.0; v.adapt.da_x_avg[c] = 0.0; v.adapt.da_g_avg[c] = 0.0;
            v.adapt.da_mu[c] = init_step_size;
            if (!v.adapt.pooled) v.adapt.wc_n[c] = 0;
            r.eps = 1.0;
        }
        v.rec[c] = r;
    }
}

template <typename T>
__global__ void copy_out_kernel(EngineView<T> v, T* q, T* p, T* g, T* U, double* eps, T* imm_user) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (i64)v.C * v.d) return;
    int c = (int)(idx / v.d), j = (int)(idx % v.d);
    i64 a = (i64)c * v.sc + (i64)j * v.sj;
    q[idx] = v.qp[a];
    if (p) p[idx] = v.pp[a];
    g[idx] = v.gp[a];
    if (imm_user) imm_user[idx] = v.imm[a];
    if (j == 0) {
        const ChainRec& r = v.rec[c];
        U[c] = (T)r.U_prop;
        eps[c] = r.eps;
        if (v.out.acceptance_probability) v.out.acceptance_probability[c] = r.accept_prob;
        if (v.out.num_doublings) v.out.num_doublings[c] = r.last_nd;
        if (v.out.is_turning) v.out.is_turning[c] = (r.last_flags & 1) ? 1 : 0;
        if (v.out.is_diverging) v.out.is_diverging[c] = (r.last_flags & 2) ? 1 : 0;
        if (v.out.n_leapfrog) v.out.n_leapfrog[c] = r.last_nleap;
        if (v.counters) {
            atomicAdd((unsigned long long*)&v.counters[0], (unsigned long long)r.total_leap);
            atomicAdd((unsigned long long*)&v.counters[1], (unsigned long long)(r.t - r.t_base));
        }
    }
}

// resume: refresh only what the caller may have changed between calls (nothing) and clear per-call counters
template <typename T>
__global__ void resume_kernel(EngineView<T> v) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= v.C) return;
    v.rec[c].total_leap = 0;
    v.rec[c].t_base = v.rec[c].t;
    if (v.rec[c].phase == PH_DONE) v.rec[c].phase = PH_START;
}

template <typename T>
static int run_typed(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                     const b2h_cfg* cfg, const b2h_adapt* adapt, void* q, void* p, void* U, void* g,
                     double* step_size, i64 C64, int n_transitions, i64 max_ticks, int resume, b2h_diag* diag,
                     void* draws, double* draw_stats, int n_store, int64_t* counters, void* ws, i64 ws_bytes,
                     bool hmc) {
    EnginePlan pl;
    int rc = make_plan(model, metric, cfg, pl, C64, max_ticks > 0);
    if (rc) return rc;
    const int C = (int)C64, d = model->dim;
    const int maxd = hmc ? 1 : cfg->max_num_expansions;
    if (!hmc && (maxd < 1 || maxd > 24)) { set_error("max_num_expansions must be in [1, 24]"); return B2H_ERR_ARG; }
    const bool adapting = adapt && adapt->enabled;
    const bool pooled = adapting && adapt->pooled;
    if (adapting && !pooled && !pl.per_chain_imm) {
        set_error("per-chain window adaptation needs a DIAG_PER_CHAIN inverse mass matrix (adapted in place)");
        return B2H_ERR_ARG;
    }
    if (adapting && (adapt->step_offset < 0 || adapt->step_offset >= adapt->num_steps)) {
        set_error("adapt.step_offset must be in [0, num_steps)");
        return B2H_ERR_ARG;
    }
    if (pl.dense && (!metric->imm || !metric->sqrt_t || !metric->chol_t)) { set_error("dense metric needs imm, sqrt_t and chol_t"); return B2H_ERR_ARG; }
    if (rng->mode == B2H_RNG_INJECTED) {
        if (!rng->z || rng->n_injected < (i64)rng->transition_offset + n_transitions || n_transitions <= 0) {
            set_error("injected draws need z and n_injected >= transition_offset + n_transitions, n_transitions > 0");
            return B2H_ERR_ARG;
        }
        if (!hmc && (!rng->u_dir || !rng->u_biased || !rng->u_uniform)) { set_error("NUTS needs u_dir/u_biased/u_uniform"); return B2H_ERR_ARG; }
        if (hmc && !rng->u_accept) { set_error("HMC needs u_accept"); return B2H_ERR_ARG; }
    }

    EngineView<T> v;
    memset(&v, 0, sizeof(v));
    size_t model_ws_bytes = pl.split ? (size_t)potential_workspace_bytes_impl(model, Num<T>::dtype, C) : 0;
    size_t model_ws_off = 0;
    size_t need = carve<T>(v, nullptr, pl, model, C, d, maxd, adapting && !pooled, model_ws_bytes, &model_ws_off);
    if (!ws || (size_t)ws_bytes < need) {
        set_error("workspace too small: need " + std::to_string(need) + " bytes");
        return B2H_ERR_WORKSPACE;
    }
    carve<T>(v, (char*)ws, pl, model, C, d, maxd, adapting && !pooled, model_ws_bytes, &model_ws_off);
    void* model_ws = model_ws_bytes ? (char*)ws + model_ws_off : nullptr;
    v.C = C; v.d = d; v.maxd = maxd;
    v.exact_doubling = cfg->exact_doubling ? 1 : 0;
    if (pl.G == 1) { v.sc = 1; v.sj = C; v.sck = 1; }
    else { v.sc = d; v.sj = 1; v.sck = (i64)maxd * d; }
    v.imm_kind = metric->kind;
    if (pl.scalar_imm) { v.imm_sc = 0; v.imm_sj = 0; }
    else if (metric->kind == B2H_IMM_DIAG) { v.imm = (T*)metric->imm; v.imm_sc = 0; v.imm_sj = 1; }
    else if (pl.per_chain_imm) { v.imm_sc = v.sc; v.imm_sj = v.sj; }
    v.rng.mode = rng->mode;
    v.rng.key.k0 = (uint32_t)rng->seed; v.rng.key.k1 = (uint32_t)(rng->seed >> 32);
    v.rng.chain_offset = rng->chain_offset; v.rng.transition_offset = rng->transition_offset;
    v.rng.n_injected = rng->n_injected;
    v.rng.z = rng->z; v.rng.u_dir = rng->u_dir; v.rng.u_biased = rng->u_biased; v.rng.u_uniform = rng->u_uniform;
    v.rng.u_accept = rng->u_accept;
    v.adapt.enabled = adapting ? 1 : 0;
    if (adapting) {
        v.adapt.pooled = pooled ? 1 : 0; v.adapt.step_offset = adapt->step_offset;
        v.adapt.num_steps = adapt->num_steps; v.adapt.stage = adapt->stage; v.adapt.window_end = adapt->window_end;
        v.adapt.target = adapt->target_acceptance_rate; v.adapt.gamma = adapt->gamma; v.adapt.t0 = adapt->t0;
        v.adapt.kappa = adapt->kappa;
        v.adapt.da_step = (i64*)adapt->da_step; v.adapt.da_x = adapt->da_x; v.adapt.da_x_avg = adapt->da_x_avg;
        v.adapt.da_g_avg = adapt->da_g_avg; v.adapt.da_mu = adapt->da_mu; v.adapt.wc_n = (i64*)adapt->wc_n;
    }
    v.out.draws = draws; v.out.draw_stats = draw_stats; v.out.n_store = n_store; v.out.thin = cfg->thin;
    if (diag) {
        v.out.acceptance_probability = diag->acceptance_probability; v.out.num_doublings = diag->num_doublings;
        v.out.is_turning = diag->is_turning; v.out.is_diverging = diag->is_diverging;
        v.out.n_leapfrog = diag->n_leapfrog;
    }
    v.div_thr = cfg->divergence_threshold;
    v.n_transitions = max_ticks > 0 ? 0 : n_transitions;
    v.hmc_L = cfg->num_integration_steps;
    v.counters = (i64*)counters;
    if (hmc && v.hmc_L < 1) { set_error("num_integration_steps must be >= 1"); return B2H_ERR_ARG; }
    if (max_ticks <= 0 && n_transitions <= 0) { set_error("need n_transitions > 0 or max_ticks > 0"); return B2H_ERR_ARG; }

    cudaStream_t st = ctx->stream;
    const i64 n = (i64)C * d;
    const int eb = 256, eg = (int)((n + eb - 1) / eb);
    if (!resume) {
        copy_in_kernel<T><<<eg, eb, 0, st>>>(v, (const T*)q, (const T*)g, (const T*)U, step_size,
                                             pl.per_chain_imm ? (const T*)metric->imm : nullptr,
                                             (T)metric->scalar, pl.scalar_imm ? 1 : 0,
                                             adapting ? adapt->initial_step_size : 0.0);
    } else {
        resume_kernel<T><<<(C + 255) / 256, 256, 0, st>>>(v);
    }
    B2H_LAUNCH_CHECK();
    int* not_done_dev = v.scratch;

    if (!pl.split) {
        rc = launch_fused_g<T>(st, v, model, max_ticks, pl.G, hmc);
    } else {
        if (pl.G == 1) { set_error("split mode needs group >= 8"); return B2H_ERR_ARG; }
        rc = run_split_g<T>(ctx, v, pl, model, metric, cfg, max_ticks, n_transitions, model_ws, model_ws_bytes,
                            not_done_dev, resume, hmc);
    }
    if (rc) return rc;
    copy_out_kernel<T><<<eg, eb, 0, st>>>(v, (T*)q, (T*)p, (T*)g, (T*)U, step_size,
                                          pl.per_chain_imm ? (T*)metric->imm : nullptr);
    B2H_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// stand-alone trajectory builders (caller-supplied tree state): the same state machine, entered after
// begin_transition (expand) or for exactly one sub-tree (integrate)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void tree_in_kernel(EngineView<T> v, b2h_tree t, const double* eps) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0 && v.imm_kind == B2H_IMM_SCALAR) {}
    if (idx >= (i64)v.C * v.d) return;
    int c = (int)(idx / v.d), j = (int)(idx % v.d);
    i64 a = (i64)c * v.sc + (i64)j * v.sj;
    v.qp[a] = ((const T*)t.proposal.q)[idx]; v.pp[a] = ((const T*)t.proposal.p)[idx]; v.gp[a] = ((const T*)t.proposal.g)[idx];
    v.ql[a] = ((const T*)t.left.q)[idx]; v.pl[a] = ((const T*)t.left.p)[idx]; v.gl[a] = ((const T*)t.left.g)[idx];
    v.qr[a] = ((const T*)t.right.q)[idx]; v.pr[a] = ((const T*)t.right.p)[idx]; v.gr[a] = ((const T*)t.right.g)[idx];
    v.msum[a] = ((const T*)t.momentum_sum)[idx];
    for (int l = 0; l < v.maxd; ++l) {
        i64 b = (i64)c * v.sck + ((i64)l * v.d + j) * v.sj;
        v.mck[b] = ((const T*)t.momentum_ckpts)[((i64)c * v.maxd + l) * v.d + j];
        v.sckp[b] = ((const T*)t.momentum_sum_ckpts)[((i64)c * v.maxd + l) * v.d + j];
    }
    if (j == 0) {
        ChainRec r;
        memset(&r, 0, sizeof(r));
        r.phase = PH_RUN;
        r.eps = eps[c];
        r.E0 = (double)((const T*)t.initial_energy)[c];
        r.U_prop = (double)((const T*)t.proposal.U)[c];
        r.E_prop = (double)((const T*)t.proposal_energy)[c];
        r.w_prop = t.proposal_weight[c];
        r.slpa_prop = t.proposal_slpa[c];
        r.U_left = (double)((const T*)t.left.U)[c];
        r.U_right = (double)((const T*)t.right.U)[c];
        r.imin = (int)t.idx_min[c]; r.imax = (int)t.idx_max[c];
        r.k = 0; r.s = 0;
        double u = draw_u(v.rng, DRAW_DIR, c, 0, 0, v.maxd);          // trajectory.py:516 for expansion 0
        r.go_right = bern(u, 0.5) ? 1 : 0;
        v.rec[c] = r;
    }
}

template <typename T>
__global__ void tree_out_kernel(EngineView<T> v, b2h_tree t) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (i64)v.C * v.d) return;
    int c = (int)(idx / v.d), j = (int)(idx % v.d);
    i64 a = (i64)c * v.sc + (i64)j * v.sj;
    ((T*)t.proposal.q)[idx] = v.qp[a]; ((T*)t.proposal.p)[idx] = v.pp[a]; ((T*)t.proposal.g)[idx] = v.gp[a];
    ((T*)t.left.q)[idx] = v.ql[a]; ((T*)t.left.p)[idx] = v.pl[a]; ((T*)t.left.g)[idx] = v.gl[a];
    ((T*)t.right.q)[idx] = v.qr[a]; ((T*)t.right.p)[idx] = v.pr[a]; ((T*)t.right.g)[idx] = v.gr[a];
    ((T*)t.momentum_sum)[idx] = v.msum[a];
    for (int l = 0; l < v.maxd; ++l) {
        i64 b = (i64)c * v.sck + ((i64)l * v.d + j) * v.sj;
        ((T*)t.momentum_ckpts)[((i64)c * v.maxd + l) * v.d + j] = v.mck[b];
        ((T*)t.momentum_sum_ckpts)[((i64)c * v.maxd + l) * v.d + j] = v.sckp[b];
    }
    if (j == 0) {
        const ChainRec& r = v.rec[c];
        ((T*)t.proposal.U)[c] = (T)r.U_prop;
        ((T*)t.proposal_energy)[c] = (T)r.E_prop;
        t.proposal_weight[c] = r.w_prop;
        t.proposal_slpa[c] = r.slpa_prop;
        ((T*)t.left.U)[c] = (T)r.U_left;
        ((T*)t.right.U)[c] = (T)r.U_right;
        t.idx_min[c] = r.imin; t.idx_max[c] = r.imax;
        if (v.out.acceptance_probability) v.out.acceptance_probability[c] = r.accept_prob;
        if (v.out.num_doublings) v.out.num_doublings[c] = r.last_nd;
        if (v.out.is_turning) v.out.is_turning[c] = (r.last_flags & 1) ? 1 : 0;
        if (v.out.is_diverging) v.out.is_diverging[c] = (r.last_flags & 2) ? 1 : 0;
        if (v.out.n_leapfrog) v.out.n_leapfrog[c] = r.last_nleap;
    }
}

template <typename T>
__global__ void subtree_in_kernel(EngineView<T> v, b2h_subtree t, const double* eps) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (i64)v.C * v.d) return;
    int c = (int)(idx / v.d), j = (int)(idx % v.d);
    i64 a = (i64)c * v.sc + (i64)j * v.sj;
    T q = ((const T*)t.state.q)[idx], p = ((const T*)t.state.p)[idx], g = ((const T*)t.state.g)[idx];
    v.ql[a] = q; v.pl[a] = p; v.gl[a] = g;
    v.qr[a] = q; v.pr[a] = p; v.gr[a] = g;
    for (int l = 0; l < v.maxd; ++l) {
        i64 b = (i64)c * v.sck + ((i64)l * v.d + j) * v.sj;
        v.mck[b] = ((const T*)t.momentum_ckpts)[((i64)c * v.maxd + l) * v.d + j];
        v.sckp[b] = ((const T*)t.momentum_sum_ckpts)[((i64)c * v.maxd + l) * v.d + j];
    }
    if (j == 0) {
        ChainRec r;
        memset(&r, 0, sizeof(r));
        r.phase = PH_RUN;
        r.eps = eps[c];
        r.E0 = (double)((const T*)t.initial_energy)[c];
        r.imin = (int)t.idx_min[c]; r.imax = (int)t.idx_max[c];
        r.k = t.expansion; r.s = 0;
        r.go_right = t.direction[c] > 0 ? 1 : 0;
        v.rec[c] = r;
    }
}

template <typename T>
__global__ void subtree_out_kernel(EngineView<T> v, b2h_subtree t) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (i64)v.C * v.d) return;
    int c = (int)(idx / v.d), j = (int)(idx % v.d);
    i64 a = (i64)c * v.sc + (i64)j * v.sj;
    const ChainRec& r = v.rec[c];
    const T* Q = r.go_right ? v.qr : v.ql; const T* P = r.go_right ? v.pr : v.pl; const T* Gd = r.go_right ? v.gr : v.gl;
    ((T*)t.state.q)[idx] = Q[a]; ((T*)t.state.p)[idx] = P[a]; ((T*)t.state.g)[idx] = Gd[a];
    ((T*)t.proposal.q)[idx] = v.qs[a]; ((T*)t.proposal.p)[idx] = v.ps[a]; ((T*)t.proposal.g)[idx] = v.gs[a];
    ((T*)t.momentum_sum)[idx] = v.sms[a];
    for (int l = 0; l < v.maxd; ++l) {
        i64 b = (i64)c * v.sck + ((i64)l * v.d + j) * v.sj;
        ((T*)t.momentum_ckpts)[((i64)c * v.maxd + l) * v.d + j] = v.mck[b];
        ((T*)t.momentum_sum_ckpts)[((i64)c * v.maxd + l) * v.d + j] = v.sckp[b];
    }
    if (j == 0) {
        ((T*)t.state.U)[c] = (T)r.U_front;
        ((T*)t.proposal.U)[c] = (T)r.U_sub;
        ((T*)t.proposal_energy)[c] = (T)r.E_sub;
        t.proposal_weight[c] = r.w_sub;
        t.proposal_slpa[c] = r.slpa_sub;
        t.idx_min[c] = r.imin; t.idx_max[c] = r.imax;
        t.trajectory_length[c] = r.sub_len;
        t.is_diverging[c] = (r.last_flags & 2) ? 1 : 0;
        t.has_terminated[c] = (r.last_flags & 4) ? 1 : 0;
    }
}

template <typename T>
__global__ void imm_in_kernel(EngineView<T> v, const T* imm_user) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (i64)v.C * v.d) return;
    const int c = (int)(idx / v.d), j = (int)(idx % v.d);
    v.imm[(i64)c * v.sc + (i64)j * v.sj] = imm_user[idx];
}

// shared set-up of the two entry points: every model, scalar / diagonal metrics (the tree state of the reference's
// closures carries no velocities, which the dense-metric engine needs)
template <typename T>
static int tree_setup(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng, const b2h_cfg* cfg,
                      i64 C64, void* ws, i64 ws_bytes, EngineView<T>& v, EnginePlan& pl, void** model_ws,
                      size_t* model_ws_bytes) {
    int rc = make_plan(model, metric, cfg, pl, C64);
    if (rc) return rc;
    if (pl.dense) { set_error("stand-alone trajectory builders need a scalar or diagonal metric (use nuts_run for a dense one)"); return B2H_ERR_UNSUPPORTED; }
    const int C = (int)C64, d = model->dim, maxd = cfg->max_num_expansions;
    if (maxd < 1 || maxd > 24) { set_error("max_num_expansions must be in [1, 24]"); return B2H_ERR_ARG; }
    memset(&v, 0, sizeof(v));
    const size_t mws = pl.split ? (size_t)potential_workspace_bytes_impl(model, Num<T>::dtype, C) : 0;
    size_t mws_off = 0;
    size_t need = carve<T>(v, nullptr, pl, model, C, d, maxd, false, mws, &mws_off);
    if (!ws || (size_t)ws_bytes < need) { set_error("workspace too small: need " + std::to_string(need) + " bytes"); return B2H_ERR_WORKSPACE; }
    carve<T>(v, (char*)ws, pl, model, C, d, maxd, false, mws, &mws_off);
    *model_ws = mws ? (char*)ws + mws_off : nullptr;
    *model_ws_bytes = mws;
    v.C = C; v.d = d; v.maxd = maxd;
    v.exact_doubling = cfg->exact_doubling ? 1 : 0;
    if (pl.G == 1) { v.sc = 1; v.sj = C; v.sck = 1; }
    else { v.sc = d; v.sj = 1; v.sck = (i64)maxd * d; }
    v.imm_kind = metric->kind;
    if (pl.scalar_imm) {
        v.imm_sc = 0; v.imm_sj = 0;
        T val = (T)metric->scalar;
        B2H_CUDA(cudaMemcpyAsync(v.imm, &val, sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        B2H_CUDA(cudaStreamSynchronize(ctx->stream));
    } else if (metric->kind == B2H_IMM_DIAG) { v.imm = (T*)metric->imm; v.imm_sc = 0; v.imm_sj = 1; }
    else {                                   // per-chain diagonal: the caller's [C x d] rows into the engine layout
        v.imm_sc = v.sc; v.imm_sj = v.sj;
        const i64 n = (i64)C * d;
        imm_in_kernel<T><<<(int)((n + 255) / 256), 256, 0, ctx->stream>>>(v, (const T*)metric->imm);
    }
    v.rng.mode = rng->mode;
    v.rng.key.k0 = (uint32_t)rng->seed; v.rng.key.k1 = (uint32_t)(rng->seed >> 32);
    v.rng.chain_offset = rng->chain_offset; v.rng.transition_offset = rng->transition_offset;
    v.rng.n_injected = rng->n_injected;
    v.rng.z = rng->z; v.rng.u_dir = rng->u_dir; v.rng.u_biased = rng->u_biased; v.rng.u_uniform = rng->u_uniform;
    v.rng.u_accept = rng->u_accept;
    v.div_thr = cfg->divergence_threshold;
    v.n_transitions = 1;
    return 0;
}

template <typename T>
static int expand_typed(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                        const b2h_cfg* cfg, b2h_tree* tree, const double* eps, i64 C, b2h_diag* diag, void* ws, i64 ws_bytes) {
    EngineView<T> v;
    EnginePlan pl;
    void* model_ws = nullptr;
    size_t model_ws_bytes = 0;
    int rc = tree_setup<T>(ctx, model, metric, rng, cfg, C, ws, ws_bytes, v, pl, &model_ws, &model_ws_bytes);
    if (rc) return rc;
    if (diag) {
        v.out.acceptance_probability = diag->acceptance_probability; v.out.num_doublings = diag->num_doublings;
        v.out.is_turning = diag->is_turning; v.out.is_diverging = diag->is_diverging; v.out.n_leapfrog = diag->n_leapfrog;
    }
    cudaStream_t st = ctx->stream;
    const i64 n = C * model->dim;
    const int eb = 256, eg = (int)((n + eb - 1) / eb);
    tree_in_kernel<T><<<eg, eb, 0, st>>>(v, *tree, eps);
    if (pl.split) rc = run_split_g<T>(ctx, v, pl, model, metric, cfg, 0, 1, model_ws, (i64)model_ws_bytes, v.scratch, 0, false);
    else rc = launch_fused_g<T>(st, v, model, 0, pl.G, false);
    if (rc) return rc;
    tree_out_kernel<T><<<eg, eb, 0, st>>>(v, *tree);
    B2H_LAUNCH_CHECK();
    return 0;
}

template <typename T>
static int subtree_typed(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                         const b2h_cfg* cfg, b2h_subtree* sub, const double* eps, i64 C, void* ws, i64 ws_bytes) {
    EngineView<T> v;
    EnginePlan pl;
    void* model_ws = nullptr;
    size_t model_ws_bytes = 0;
    int rc = tree_setup<T>(ctx, model, metric, rng, cfg, C, ws, ws_bytes, v, pl, &model_ws, &model_ws_bytes);
    if (rc) return rc;
    if (sub->max_num_steps < 1 || sub->expansion < 0 ||
        ((i64)1 << sub->expansion) - 1 + sub->max_num_steps > ((i64)1 << cfg->max_num_expansions) - 1) {
        set_error("sub-tree: the uniform-draw slots 2**expansion - 1 + step must fit 2**max_num_expansions - 1");
        return B2H_ERR_ARG;
    }
    v.sub_max_steps = sub->max_num_steps;
    v.stop_at_subtree_end = 1;
    cudaStream_t st = ctx->stream;
    const i64 n = C * model->dim;
    const int eb = 256, eg = (int)((n + eb - 1) / eb);
    subtree_in_kernel<T><<<eg, eb, 0, st>>>(v, *sub, eps);
    if (pl.split) rc = run_split_g<T>(ctx, v, pl, model, metric, cfg, 0, 1, model_ws, (i64)model_ws_bytes, v.scratch, 0, false);
    else rc = launch_fused_g<T>(st, v, model, 0, pl.G, false);
    if (rc) return rc;
    subtree_out_kernel<T><<<eg, eb, 0, st>>>(v, *sub);
    B2H_LAUNCH_CHECK();
    return 0;
}

int nuts_expand_impl(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                     const b2h_cfg* cfg, b2h_tree* tree, const double* eps, i64 C, b2h_diag* diag, void* ws, i64 ws_bytes) {
    if (!ctx || !model || !metric || !rng || !cfg || !tree || !eps) { set_error("null argument"); return B2H_ERR_ARG; }
    if (cfg->dtype == B2H_F64) return expand_typed<double>(ctx, model, metric, rng, cfg, tree, eps, C, diag, ws, ws_bytes);
    if (cfg->dtype == B2H_F32) return expand_typed<float>(ctx, model, metric, rng, cfg, tree, eps, C, diag, ws, ws_bytes);
    set_error("bad dtype");
    return B2H_ERR_ARG;
}

int nuts_subtree_impl(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                      const b2h_cfg* cfg, b2h_subtree* sub, const double* eps, i64 C, void* ws, i64 ws_bytes) {
    if (!ctx || !model || !metric || !rng || !cfg || !sub || !eps) { set_error("null argument"); return B2H_ERR_ARG; }
    if (cfg->dtype == B2H_F64) return subtree_typed<double>(ctx, model, metric, rng, cfg, sub, eps, C, ws, ws_bytes);
    if (cfg->dtype == B2H_F32) return subtree_typed<float>(ctx, model, metric, rng, cfg, sub, eps, C, ws, ws_bytes);
    set_error("bad dtype");
    return B2H_ERR_ARG;
}

int nuts_run_impl(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                  const b2h_cfg* cfg, const b2h_adapt* adapt, void* q, void* p, void* U, void* g, double* step_size,
                  i64 C, int n_transitions, i64 max_ticks, int resume, b2h_diag* diag, void* draws,
                  double* draw_stats, int n_store, int64_t* counters, void* ws, i64 ws_bytes, bool hmc) {
    if (!ctx || !model || !metric || !rng || !cfg || !q || !U || !g || !step_size) {
        set_error("null argument");
        return B2H_ERR_ARG;
    }
    if (C <= 0 || C > (1ll << 30) || model->dim <= 0) { set_error("bad C or dim"); return B2H_ERR_ARG; }
    if (cfg->dtype == B2H_F64)
        return run_typed<double>(ctx, model, metric, rng, cfg, adapt, q, p, U, g, step_size, C, n_transitions,
                                 max_ticks, resume, diag, draws, draw_stats, n_store, counters, ws, ws_bytes, hmc);
    if (cfg->dtype == B2H_F32)
        return run_typed<float>(ctx, model, metric, rng, cfg, adapt, q, p, U, g, step_size, C, n_transitions,
                                max_ticks, resume, diag, draws, draw_stats, n_store, counters, ws, ws_bytes, hmc);
    set_error("dtype must be B2H_F32 or B2H_F64");
    return B2H_ERR_ARG;
}

int engine_plan_group(const b2h_model* model, const b2h_metric* metric, const b2h_cfg* cfg, i64 C, bool free_running) {
    EnginePlan pl;
    if (make_plan(model, metric, cfg, pl, C, free_running)) return -1;
    return pl.G;
}

i64 engine_workspace_bytes(const b2h_model* model, const b2h_metric* metric, const b2h_cfg* cfg, i64 C) {
    EnginePlan pl;
    if (make_plan(model, metric, cfg, pl, C)) return -1;
    const int maxd = cfg->max_num_expansions > 0 ? cfg->max_num_expansions : 1;
    size_t mws = pl.split ? (size_t)potential_workspace_bytes_impl(model, cfg->dtype, C) : 0;
    if (cfg->dtype == B2H_F64) {
        EngineView<double> v;
        return (i64)carve<double>(v, nullptr, pl, model, (int)C, model->dim, maxd, true, mws, nullptr);
    }
    EngineView<float> v;
    return (i64)carve<float>(v, nullptr, pl, model, (int)C, model->dim, maxd, true, mws, nullptr);
}

}  // namespace b2h
