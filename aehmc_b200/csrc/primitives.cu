// Batched primitives behind the reference's L1 closures (SURVEY.md section 8a):
// potential/gradient, metric (momentum, kinetic energy, U-turn test), the fused
// velocity-Verlet integrator, iterative U-turn checkpoints, adaptation algorithms.
// Row-major [C x d] arrays, one warp (or sub-warp group) per chain, 128-bit
// vectorised where rows are 16-byte aligned.
#include "engine.cuh"
#include "launch.h"
#include "models.cuh"

namespace b2h {

static ModelDev to_dev(const b2h_model* m) {
    ModelDev d;
    d.kind = m->kind; d.dim = m->dim; d.n_data = m->n_data;
    d.a = m->a; d.b = m->b; d.c = m->c; d.s0 = m->s0; d.s1 = m->s1;
    return d;
}

template <int G>
struct PGeo {
    static constexpr int kThreads = 128;
    static constexpr int kChainsPerBlock = 128 / G;
    __device__ static i64 chain() { return (i64)blockIdx.x * kChainsPerBlock + threadIdx.x / G; }
    static int grid(i64 C) { return (int)((C + kChainsPerBlock - 1) / kChainsPerBlock); }
};

// ---------------------------------------------------------------------------
// potential and gradient (hmc.new_state, hmc.py:16-40)
// ---------------------------------------------------------------------------
template <typename T, int G, int MODEL>
__global__ void __launch_bounds__(128) potential_grad_kernel(ModelDev m, const T* q, T* U, T* g, i64 C) {
    const i64 c = PGeo<G>::chain();
    if (c >= C) return;
    const int lane = Group<G>::lane();
    T u = model_grad<T, G, MODEL>(m, q + c * m.dim, g + c * m.dim, 1, lane, nullptr);
    if (lane == 0) U[c] = u;
}

// U[c] = 0.5 * sum_j (q - mu)_j g_j  (correlated Gaussian, after the precision GEMM)
template <typename T>
__global__ void __launch_bounds__(128) corr_potential_kernel(const T* q, const T* mu, const T* g, T* U, i64 C, int d) {
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    T acc = 0;
    for (int j = lane; j < d; j += 32) acc += (q[c * d + j] - mu[j]) * g[c * d + j];
    double s = Group<32>::sum1((double)acc, nullptr);
    if (lane == 0) U[c] = (T)0.5 * (T)s;
}

template <typename T>
int potential_and_grad_impl(b2h_ctx* ctx, const b2h_model* model, const T* q, T* U, T* g, i64 C, void* ws,
                            i64 ws_bytes, bool gradient_only) {
    cudaStream_t st = ctx->stream;
    ModelDev m = to_dev(model);
    const int d = model->dim;
    switch (model->kind) {
        case B2H_MODEL_IID_GAUSSIAN:
            if (d <= 64) potential_grad_kernel<T, 8, MODEL_IID><<<PGeo<8>::grid(C), 128, 0, st>>>(m, q, U, g, C);
            else potential_grad_kernel<T, 32, MODEL_IID><<<PGeo<32>::grid(C), 128, 0, st>>>(m, q, U, g, C);
            break;
        case B2H_MODEL_FUNNEL:
            if (d < 2) { set_error("funnel needs dim >= 2"); return B2H_ERR_ARG; }
            potential_grad_kernel<T, 8, MODEL_FUNNEL><<<PGeo<8>::grid(C), 128, 0, st>>>(m, q, U, g, C);
            break;
        case B2H_MODEL_EIGHT_SCHOOLS:
            if (d < 3) { set_error("eight schools needs dim >= 3"); return B2H_ERR_ARG; }
            potential_grad_kernel<T, 8, MODEL_SCHOOLS><<<PGeo<8>::grid(C), 128, 0, st>>>(m, q, U, g, C);
            break;
        case B2H_MODEL_CORR_GAUSSIAN:
            launch_dense_apply<T>(st, q, (const T*)model->b, g, (int)C, d, d, nullptr, (const T*)model->a);
            if (!gradient_only) corr_potential_kernel<T><<<PGeo<32>::grid(C), 128, 0, st>>>(q, (const T*)model->a, g, U, C, d);
            break;
        case B2H_MODEL_LOGISTIC:
            return logistic_potential_and_grad<T>(ctx, model, q, U, g, C, ws, ws_bytes, 0);
        case B2H_MODEL_USER:
            return user_potential_and_grad<T>(ctx, model, q, U, g, C, ws, ws_bytes);
        default:
            set_error("unknown model kind");
            return B2H_ERR_ARG;
    }
    B2H_LAUNCH_CHECK();
    return 0;
}
template int potential_and_grad_impl<float>(b2h_ctx*, const b2h_model*, const float*, float*, float*, i64, void*, i64, bool);
template int potential_and_grad_impl<double>(b2h_ctx*, const b2h_model*, const double*, double*, double*, i64, void*,
                                             i64, bool);

i64 potential_workspace_bytes_impl(const b2h_model* m, int dtype, i64 C) {
    if (m->kind == B2H_MODEL_LOGISTIC) return logistic_workspace_bytes(m, dtype, C);
    if (m->kind == B2H_MODEL_USER) return user_workspace_bytes(m, dtype, C);
    return 0;
}

// ---------------------------------------------------------------------------
// metric helpers
// ---------------------------------------------------------------------------
struct ImmView {
    const void* imm;
    i64 sc, sj;      // imm(c, j) = imm[c*sc + j*sj]
    double scalar;
    int kind;
};

static ImmView imm_view(const b2h_metric* m, i64 d) {
    ImmView v;
    v.imm = m->imm; v.scalar = m->scalar; v.kind = m->kind;
    v.sc = m->kind == B2H_IMM_DIAG_PER_CHAIN ? d : 0;
    v.sj = (m->kind == B2H_IMM_DIAG || m->kind == B2H_IMM_DIAG_PER_CHAIN) ? 1 : 0;
    return v;
}

static bool is_dense(const b2h_metric* m) { return m->kind == B2H_IMM_DENSE || m->kind == B2H_IMM_DENSE_PER_CHAIN; }

// out = in . M of a dense metric: the shared [d x d] matrix through the dense contraction, per-chain [C x d x d]
// matrices through the batched per-chain product (tri applies to the latter; the shared path reads M in full)
template <typename T>
static void metric_apply(cudaStream_t st, const b2h_metric* m, const T* in, const void* M, T* out, i64 C, int d, int tri) {
    if (m->kind == B2H_IMM_DENSE_PER_CHAIN) launch_dense_apply_pc<T>(st, in, (const T*)M, out, C, d, tri);
    else launch_dense_apply<T>(st, in, (const T*)M, out, (int)C, d, d, nullptr, nullptr);
}

static int check_metric(const b2h_metric* m, i64 d) {
    if (m->kind != B2H_IMM_DENSE_PER_CHAIN) return 0;
    if (!m->imm || !m->sqrt_t || !m->chol_t) { set_error("per-chain dense metric needs imm, sqrt_t and chol_t"); return B2H_ERR_ARG; }
    if (d < 1 || d > B2H_DENSE_PER_CHAIN_MAX_DIM) {
        set_error("a per-chain dense metric needs 1 <= d <= " + std::to_string(B2H_DENSE_PER_CHAIN_MAX_DIM) +
                  " (B2H_DENSE_PER_CHAIN_MAX_DIM); for larger d adapt one shared dense matrix (pooled=True)");
        return B2H_ERR_ARG;
    }
    return 0;
}

template <typename T>
B2H_DEVINL T imm_at(const ImmView& v, i64 c, int j) {
    if (v.kind == B2H_IMM_SCALAR) return (T)v.scalar;
    return ((const T*)v.imm)[c * v.sc + (i64)j * v.sj];
}

// K[c] = 0.5 sum (imm p) p  (metrics.py:70-73).  vel != nullptr: dense, vel = p . imm
template <typename T>
__global__ void __launch_bounds__(128) kinetic_kernel(ImmView iv, const T* p, const T* vel, T* K, i64 C, int d) {
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    T acc = 0;
    for (int j = lane; j < d; j += 32) {
        T pj = p[c * d + j];
        T v = vel ? vel[c * d + j] : imm_at<T>(iv, c, j) * pj;
        acc += v * pj;
    }
    double s = Group<32>::sum1((double)acc, nullptr);
    if (lane == 0) K[c] = (T)0.5 * (T)s;
}

// is_turning (metrics.py:75-104)
template <typename T>
__global__ void __launch_bounds__(128) turning_kernel(ImmView iv, const T* pl, const T* pr, const T* ps,
                                                      const T* vl, const T* vr, uint8_t* out, i64 C, int d) {
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    T dl = 0, dr = 0;
    for (int j = lane; j < d; j += 32) {
        i64 a = c * d + j;
        T l = pl[a], r = pr[a];
        T rho = ps[a] - (r + l) / (T)2;
        T im = vl ? (T)0 : imm_at<T>(iv, c, j);
        T vleft = vl ? vl[a] : im * l, vright = vr ? vr[a] : im * r;
        dl += vleft * rho;
        dr += vright * rho;
    }
    double red[2] = {(double)dl, (double)dr};
    Group<32>::sum<2>(red, nullptr);
    if (lane == 0) out[c] = ((T)red[0] <= (T)0 || (T)red[1] <= (T)0) ? 1 : 0;
}

// momentum (metrics.py:65-68): diag family p = sqrt(1/imm) z ; dense: z only (GEMM follows)
template <typename T>
__global__ void momentum_kernel(ImmView iv, RngView rng, T* p, i64 C, int d, int transition, int dense) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * d) return;
    i64 c = idx / d;
    int j = (int)(idx % d);
    T z = (T)draw_z(rng, (int)c, transition, j, d);
    p[idx] = dense ? z : sqrt((T)1 / imm_at<T>(iv, c, j)) * z;
}

// ---------------------------------------------------------------------------
// fused velocity Verlet for elementwise targets (integrators.py:58-73), n_steps in one launch.
// Warp per chain, VEC elements per 128-bit access; q, p, g stay in registers across steps when
// the row fits (d <= 32*VEC*REGS), otherwise they stream through global memory.
// ---------------------------------------------------------------------------
template <typename T, int MODEL>
__global__ void __launch_bounds__(128)
leapfrog_fused_kernel(ModelDev m, ImmView iv, T* q, T* p, T* U, T* g, const double* eps, const int8_t* dir,
                      int n_steps, i64 C) {
    constexpr int G = 32;
    const i64 c = PGeo<G>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const int d = m.dim;
    T* qc = q + c * d; T* pc = p + c * d; T* gc = g + c * d;
    const T e = (T)(eps[c] * (dir ? (double)dir[c] : 1.0));
    const T he = (T)0.5 * e;
    T u = U[c];
    for (int s = 0; s < n_steps; ++s) {
        for (int j = lane; j < d; j += G) {
            T ph = pc[j] - he * gc[j];
            pc[j] = ph;
            qc[j] = qc[j] + e * (imm_at<T>(iv, c, j) * ph);
        }
        __syncwarp();
        u = model_grad<T, G, MODEL>(m, qc, gc, 1, lane, nullptr);
        __syncwarp();
        for (int j = lane; j < d; j += G) pc[j] = pc[j] - he * gc[j];
    }
    if (lane == 0) U[c] = u;
}

// 128-bit vectorised single-pass variant for the iid Gaussian (pure elementwise gradient):
// every element is read once and written once per launch regardless of n_steps.
template <typename T, int VEC>
struct alignas(sizeof(T) * VEC) Pack { T v[VEC]; };

template <typename T, int VEC>
__global__ void __launch_bounds__(128)
leapfrog_iid_vec_kernel(ModelDev m, ImmView iv, T* q, T* p, T* U, T* g, const double* eps, const int8_t* dir,
                        int n_steps, i64 C) {
    typedef Pack<T, VEC> P;
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const int d = m.dim, nv = d / VEC;
    const T e = (T)(eps[c] * (dir ? (double)dir[c] : 1.0));
    const T he = (T)0.5 * e;
    const T* mu = (const T*)m.a;
    const T* ivar = (const T*)m.b;
    P* qv = (P*)(q + c * d); P* pv = (P*)(p + c * d); P* gv = (P*)(g + c * d);
    T acc = 0;
    for (int k = lane; k < nv; k += 32) {
        P Q = qv[k], Pm = pv[k], Gd = gv[k];
        P Mu = ((const P*)mu)[k], Iv = ((const P*)ivar)[k];
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            T im = imm_at<T>(iv, c, k * VEC + i);
            T qq = Q.v[i], pp = Pm.v[i], gg = Gd.v[i], r = 0;
            for (int s = 0; s < n_steps; ++s) {
                T ph = pp - he * gg;
                qq = qq + e * (im * ph);
                r = qq - Mu.v[i];
                gg = r * Iv.v[i];
                pp = ph - he * gg;
            }
            Q.v[i] = qq; Pm.v[i] = pp; Gd.v[i] = gg;
            if (n_steps > 0) acc += r * gg;
        }
        qv[k] = Q; pv[k] = Pm; gv[k] = Gd;
    }
    double s = Group<32>::sum1((double)acc, nullptr);
    if (lane == 0 && n_steps > 0) U[c] = (T)0.5 * (T)s + (T)m.s0;
}

// split-path elementwise pieces (any model / metric)
template <typename T>
__global__ void halfkick_kernel(ImmView iv, T* q, T* p, const T* g, const double* eps, const int8_t* dir, i64 C, int d,
                                int drift) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * d) return;
    i64 c = idx / d;
    int j = (int)(idx % d);
    const T e = (T)(eps[c] * (dir ? (double)dir[c] : 1.0));
    T ph = p[idx] - (T)0.5 * e * g[idx];
    p[idx] = ph;
    if (drift) q[idx] = q[idx] + e * (imm_at<T>(iv, c, j) * ph);
}

template <typename T>
__global__ void drift_kernel(T* q, const T* vel, const double* eps, const int8_t* dir, i64 C, int d) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * d) return;
    i64 c = idx / d;
    const T e = (T)(eps[c] * (dir ? (double)dir[c] : 1.0));
    q[idx] = q[idx] + e * vel[idx];
}

template <typename T>
__global__ void kick_kernel(T* p, const T* g, const double* eps, const int8_t* dir, i64 C, int d) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * d) return;
    i64 c = idx / d;
    const T e = (T)(eps[c] * (dir ? (double)dir[c] : 1.0));
    p[idx] = p[idx] - (T)0.5 * e * g[idx];
}

template <typename T>
static int leapfrog_typed(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, T* q, T* p, T* U, T* g,
                          const double* eps, const int8_t* dir, int n_steps, i64 C, void* ws, i64 ws_bytes) {
    cudaStream_t st = ctx->stream;
    const int d = model->dim;
    ImmView iv = imm_view(metric, d);
    ModelDev m = to_dev(model);
    const bool dense = is_dense(metric);
    if (int rc = check_metric(metric, d)) return rc;
    const bool fused = !dense && (model->kind == B2H_MODEL_IID_GAUSSIAN || model->kind == B2H_MODEL_FUNNEL ||
                                  model->kind == B2H_MODEL_EIGHT_SCHOOLS);
    if (fused) {
        const int grid = PGeo<32>::grid(C);
        constexpr int VEC = 16 / sizeof(T);
        auto aligned = [](const void* x) { return ((uintptr_t)x & 15) == 0; };
        if (model->kind == B2H_MODEL_IID_GAUSSIAN && d % VEC == 0 && aligned(q) && aligned(p) && aligned(g) &&
            aligned(model->a) && aligned(model->b)) {
            leapfrog_iid_vec_kernel<T, VEC><<<grid, 128, 0, st>>>(m, iv, q, p, U, g, eps, dir, n_steps, C);
        } else if (model->kind == B2H_MODEL_IID_GAUSSIAN) {
            leapfrog_fused_kernel<T, MODEL_IID><<<grid, 128, 0, st>>>(m, iv, q, p, U, g, eps, dir, n_steps, C);
        } else if (model->kind == B2H_MODEL_FUNNEL) {
            leapfrog_fused_kernel<T, MODEL_FUNNEL><<<grid, 128, 0, st>>>(m, iv, q, p, U, g, eps, dir, n_steps, C);
        } else {
            leapfrog_fused_kernel<T, MODEL_SCHOOLS><<<grid, 128, 0, st>>>(m, iv, q, p, U, g, eps, dir, n_steps, C);
        }
        B2H_LAUNCH_CHECK();
        return 0;
    }
    // split path: dense metric and/or contraction gradients
    const i64 n = C * d;
    const int eb = 256, eg = (int)((n + eb - 1) / eb);
    i64 mws = potential_workspace_bytes_impl(model, Num<T>::dtype, C);
    i64 need = mws + (dense ? (i64)n * (i64)sizeof(T) + 256 : 0);
    if (need > 0 && (!ws || ws_bytes < need)) {
        set_error("leapfrog workspace too small: need " + std::to_string(need) + " bytes");
        return B2H_ERR_WORKSPACE;
    }
    T* vel = dense ? (T*)ws : nullptr;
    void* model_ws = dense ? (void*)((char*)ws + (((size_t)n * sizeof(T) + 255) & ~(size_t)255)) : ws;
    for (int s = 0; s < n_steps; ++s) {
        halfkick_kernel<T><<<eg, eb, 0, st>>>(iv, q, p, g, eps, dir, C, d, dense ? 0 : 1);
        if (dense) {
            metric_apply<T>(st, metric, p, metric->imm, vel, C, d, 0);
            drift_kernel<T><<<eg, eb, 0, st>>>(q, vel, eps, dir, C, d);
        }
        int rc = potential_and_grad_impl<T>(ctx, model, q, U, g, C, model_ws, mws);
        if (rc) return rc;
        kick_kernel<T><<<eg, eb, 0, st>>>(p, g, eps, dir, C, d);
    }
    B2H_LAUNCH_CHECK();
    return 0;
}

// ---------------------------------------------------------------------------
// iterative U-turn primitives (termination.py:85-187, 192-235), diag-family metrics
// ---------------------------------------------------------------------------
__global__ void storage_indices_kernel(const int64_t* step, int64_t* imin, int64_t* imax, i64 n) {
    i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int a, b;
    storage_indices((int)step[i], a, b);
    imin[i] = a; imax[i] = b;
}

template <typename T>
__global__ void __launch_bounds__(128)
termination_update_kernel(T* mck, T* sck, int64_t* imin, int64_t* imax, const T* msum, const T* mom,
                          const int64_t* step, i64 C, int d, int maxd) {
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const int s = (int)step[c];
    int lo, hi;
    if (s == 0) { lo = (int)imin[c]; hi = (int)imax[c]; }        // stale indices (Q2)
    else storage_indices(s, lo, hi);
    if ((s & 1) == 0 && hi >= 0 && hi < maxd) {
        for (int j = lane; j < d; j += 32) {
            i64 b = (c * maxd + hi) * d + j;
            mck[b] = mom[c * d + j];
            sck[b] = msum[c * d + j];
        }
    }
    __syncwarp();
    if (lane == 0) { imin[c] = lo; imax[c] = hi; }
}

template <typename T>
__global__ void __launch_bounds__(128)
iterative_turning_kernel(ImmView iv, const T* mck, const T* sck, const int64_t* imin, const int64_t* imax,
                         const T* msum, const T* mom, uint8_t* out, i64 C, int d, int maxd) {
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const int lo = (int)imin[c], hi = (int)imax[c];
    bool term = false;
    if (hi >= lo) {
        for (int i = hi; i >= lo; --i) {
            T dl = 0, dr = 0;
            for (int j = lane; j < d; j += 32) {
                i64 a = c * d + j, b = (c * maxd + i) * d + j;
                T mm = mck[b], p = mom[a];
                T subsum = msum[a] - sck[b] + mm;
                T rho = subsum - (p + mm) / (T)2;
                T im = imm_at<T>(iv, c, j);
                dl += (im * mm) * rho;
                dr += (im * p) * rho;
            }
            double red[2] = {(double)dl, (double)dr};
            Group<32>::sum<2>(red, nullptr);
            if ((T)red[0] <= (T)0 || (T)red[1] <= (T)0) { term = true; break; }
        }
    }
    if (lane == 0) out[c] = term ? 1 : 0;
}

// ---------------------------------------------------------------------------
// 128-bit vectorised variants of the metric / U-turn primitives (warp per chain, lane = one 16-byte chunk, two
// chunks in flight per array): used when the rows are 16-byte aligned and the metric is scalar or has unit stride.
// ---------------------------------------------------------------------------
template <typename T> struct V16;
template <> struct V16<double> { static constexpr int N = 2; using type = double2; };
template <> struct V16<float> { static constexpr int N = 4; using type = float4; };

template <typename T>
B2H_DEVINL void ld16(const T* p, T (&v)[V16<T>::N]) {
    const typename V16<T>::type w = *reinterpret_cast<const typename V16<T>::type*>(p);
    const T* e = reinterpret_cast<const T*>(&w);
#pragma unroll
    for (int i = 0; i < V16<T>::N; ++i) v[i] = e[i];
}
template <typename T>
B2H_DEVINL void st16(T* p, const T (&v)[V16<T>::N]) {
    typename V16<T>::type w;
    T* e = reinterpret_cast<T*>(&w);
#pragma unroll
    for (int i = 0; i < V16<T>::N; ++i) e[i] = v[i];
    *reinterpret_cast<typename V16<T>::type*>(p) = w;
}
template <typename T>
B2H_DEVINL void imm16(const ImmView& iv, i64 c, int j, T (&v)[V16<T>::N]) {
    if (iv.kind == B2H_IMM_SCALAR) {
#pragma unroll
        for (int i = 0; i < V16<T>::N; ++i) v[i] = (T)iv.scalar;
    } else {
        ld16<T>((const T*)iv.imm + c * iv.sc + j, v);
    }
}
static bool vec_ok(const ImmView& iv, i64 d, int dtype, std::initializer_list<const void*> ptrs) {
    const int n = 16 / (int)dtype_size(dtype);
    if (d % n) return false;
    if (iv.kind != B2H_IMM_SCALAR && (iv.sj != 1 || ((uintptr_t)iv.imm & 15) || (iv.sc % n))) return false;
    for (const void* p : ptrs)
        if (p && ((uintptr_t)p & 15)) return false;
    return true;
}

template <typename T>
__global__ void __launch_bounds__(128) kinetic_vec_kernel(ImmView iv, const T* p, const T* vel, T* K, i64 C, int d) {
    constexpr int N = V16<T>::N;
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    T acc = 0;
#pragma unroll 2
    for (int j = lane * N; j < d; j += 32 * N) {
        T pj[N], vj[N];
        ld16<T>(p + c * d + j, pj);
        if (vel) ld16<T>(vel + c * d + j, vj);
        else imm16<T>(iv, c, j, vj);
#pragma unroll
        for (int i = 0; i < N; ++i) acc += (vel ? vj[i] : vj[i] * pj[i]) * pj[i];
    }
    double s = Group<32>::sum1((double)acc, nullptr);
    if (lane == 0) K[c] = (T)0.5 * (T)s;
}

template <typename T>
__global__ void __launch_bounds__(128) turning_vec_kernel(ImmView iv, const T* pl, const T* pr, const T* ps, const T* vl,
                                                          const T* vr, uint8_t* out, i64 C, int d) {
    constexpr int N = V16<T>::N;
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    T dl = 0, dr = 0;
#pragma unroll 2
    for (int j = lane * N; j < d; j += 32 * N) {
        const i64 a = c * d + j;
        T l[N], r[N], sm[N], a0[N], a1[N];
        ld16<T>(pl + a, l); ld16<T>(pr + a, r); ld16<T>(ps + a, sm);
        if (vl) { ld16<T>(vl + a, a0); ld16<T>(vr + a, a1); }
        else imm16<T>(iv, c, j, a0);
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const T rho = sm[i] - (r[i] + l[i]) / (T)2;
            const T vleft = vl ? a0[i] : a0[i] * l[i], vright = vl ? a1[i] : a0[i] * r[i];
            dl += vleft * rho;
            dr += vright * rho;
        }
    }
    double red[2] = {(double)dl, (double)dr};
    Group<32>::sum<2>(red, nullptr);
    if (lane == 0) out[c] = ((T)red[0] <= (T)0 || (T)red[1] <= (T)0) ? 1 : 0;
}

template <typename T>
__global__ void __launch_bounds__(128)
termination_update_vec_kernel(T* mck, T* sck, int64_t* imin, int64_t* imax, const T* msum, const T* mom,
                              const int64_t* step, i64 C, int d, int maxd) {
    constexpr int N = V16<T>::N;
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const int s = (int)step[c];
    int lo, hi;
    if (s == 0) { lo = (int)imin[c]; hi = (int)imax[c]; }        // stale indices (Q2)
    else storage_indices(s, lo, hi);
    if ((s & 1) == 0 && hi >= 0 && hi < maxd) {
#pragma unroll 2
        for (int j = lane * N; j < d; j += 32 * N) {
            const i64 b = (c * maxd + hi) * d + j;
            T m[N], ms[N];
            ld16<T>(mom + c * d + j, m); ld16<T>(msum + c * d + j, ms);
            st16<T>(mck + b, m); st16<T>(sck + b, ms);
        }
    }
    __syncwarp();
    if (lane == 0) { imin[c] = lo; imax[c] = hi; }
}

template <typename T>
__global__ void __launch_bounds__(128)
iterative_turning_vec_kernel(ImmView iv, const T* mck, const T* sck, const int64_t* imin, const int64_t* imax,
                             const T* msum, const T* mom, uint8_t* out, i64 C, int d, int maxd) {
    constexpr int N = V16<T>::N;
    const i64 c = PGeo<32>::chain();
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const int lo = (int)imin[c], hi = (int)imax[c];
    bool term = false;
    if (hi >= lo) {
        for (int i = hi; i >= lo; --i) {
            T dl = 0, dr = 0;
#pragma unroll 2
            for (int j = lane * N; j < d; j += 32 * N) {
                const i64 a = c * d + j, b = (c * maxd + i) * d + j;
                T mm[N], pp[N], ss[N], sc[N], im[N];
                ld16<T>(mck + b, mm); ld16<T>(sck + b, sc); ld16<T>(mom + a, pp); ld16<T>(msum + a, ss);
                imm16<T>(iv, c, j, im);
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const T subsum = ss[k] - sc[k] + mm[k];
                    const T rho = subsum - (pp[k] + mm[k]) / (T)2;
                    dl += (im[k] * mm[k]) * rho;
                    dr += (im[k] * pp[k]) * rho;
                }
            }
            double red[2] = {(double)dl, (double)dr};
            Group<32>::sum<2>(red, nullptr);
            if ((T)red[0] <= (T)0 || (T)red[1] <= (T)0) { term = true; break; }
        }
    }
    if (lane == 0) out[c] = term ? 1 : 0;
}

// ---------------------------------------------------------------------------
// adaptation algorithms (algorithms.py:79-115,166-202; mass_matrix.py:81-118)
// ---------------------------------------------------------------------------
__global__ void dual_averaging_kernel(const double* p_accept, double target, double gamma, double t0, double kappa,
                                      int64_t* step, double* x, double* x_avg, double* g_avg, const double* mu, i64 C) {
    i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double st = (double)step[c];
    double grad = target - p_accept[c];
    double eta = 1.0 / (st + t0);
    double ng = (1.0 - eta) * g_avg[c] + eta * grad;
    double nx = mu[c] - (sqrt(st) / gamma) * ng;
    double xe = pow(st, -kappa);
    double nxa = xe * x[c] + (1.0 - xe) * x_avg[c];
    step[c] += 1; x[c] = nx; x_avg[c] = nxa; g_avg[c] = ng;
}

template <typename T>
__global__ void welford_kernel(const T* value, T* mean, T* m2, int64_t* n, i64 C, int d, int full) {
    // one block per chain; diag: thread per j; full: threads over (i, j) with a two-phase update
    const i64 c = blockIdx.x;
    const i64 nn = n[c] + 1;
    extern __shared__ unsigned char smem_raw[];
    T* delta = (T*)smem_raw;          // [d]
    T* udelta = delta + d;            // [d]
    for (int j = threadIdx.x; j < d; j += blockDim.x) {
        T val = value[c * d + j];
        T dl = val - mean[c * d + j];
        T mn = mean[c * d + j] + dl / (T)nn;
        delta[j] = dl;
        udelta[j] = val - mn;
        mean[c * d + j] = mn;
        if (!full) m2[c * d + j] = m2[c * d + j] + (val - mn) * dl;
    }
    __syncthreads();
    if (full) {
        for (i64 k = threadIdx.x; k < (i64)d * d; k += blockDim.x) {
            int i = (int)(k / d), j = (int)(k % d);
            m2[c * d * d + k] = m2[c * d * d + k] + udelta[i] * delta[j];   // outer(updated_delta, delta)
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) n[c] = nn;
}

template <typename T>
__global__ void mass_matrix_final_kernel(const T* m2, const int64_t* n, T* out, i64 C, int d, int full) {
    i64 per = full ? (i64)d * d : d;
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * per) return;
    i64 c = idx / per, k = idx % per;
    double nn = (double)n[c];
    T cov = m2[idx] / (T)(nn - 1.0);
    T scaled = (T)(nn / (nn + 5.0)) * cov;
    T shrink = (T)(1e-3 * (5.0 / (nn + 5.0)));
    bool on_diag = !full || (k / d == k % d);
    out[idx] = scaled + (on_diag ? shrink : (T)0);
}

// ---------------------------------------------------------------------------
// proposal scalars (proposals.py:41-52, 96-100, 130-174)
// ---------------------------------------------------------------------------
template <typename T>
__global__ void proposal_update_kernel(const T* E0, const T* U, const T* K, double thr, T* energy, double* weight,
                                       double* lpa, uint8_t* div, i64 C) {
    i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    T e = U[c] + K[c];
    double delta = (double)(E0[c] - e);
    if (isnan(delta)) delta = -INFINITY;
    energy[c] = e;
    weight[c] = delta;
    lpa[c] = delta > 0 ? 0.0 : delta;
    div[c] = fabs(delta) > thr ? 1 : 0;
}

__global__ void progressive_sampling_kernel(int biased, const double* w_old, const double* w_new, const double* s_old,
                                            const double* s_new, const double* u, uint8_t* acc, double* w_out,
                                            double* s_out, i64 C) {
    i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    double p;
    if (biased) p = fmin(fmax(exp(w_new[c] - w_old[c]), 0.0), 1.0);
    else { p = expit(w_new[c] - w_old[c]); if (isnan(p)) p = 0.0; }
    acc[c] = bern(u[c], p) ? 1 : 0;
    w_out[c] = lae(w_old[c], w_new[c]);
    s_out[c] = lae(s_old[c], s_new[c]);
}

template <typename T>
__global__ void select_rows_kernel(const uint8_t* mask, const T* a, const T* b, T* out, i64 C, int d) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * d) return;
    out[idx] = mask[idx / d] ? a[idx] : b[idx];
}

// hmc_proposal.propose after the integration (hmc.py:183-204): one warp per chain.  The integrated state gets its
// momentum flipped; energies E = U + K (K(-p) = K(p)); delta = E_old - E_new (NaN -> -inf); diverging = |delta| >
// threshold (Q15: a divergent transition is NOT force-rejected); p_accept = clip(exp(delta), 0, 1); accept from the
// uniform with numpy's binomial(1, p) rule; the final state overwrites the `new` arrays.
template <typename T>
__global__ void __launch_bounds__(128)
hmc_accept_kernel(const T* q0, const T* p0, const T* g0, const T* U0, T* q1, T* p1, T* g1, T* U1, const T* K0,
                  const T* K1, const double* u, double thr, double* p_accept, uint8_t* diverging, i64 C, int d) {
    const i64 c = (i64)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (c >= C) return;
    const int lane = threadIdx.x & 31;
    const T E0 = U0[c] + K0[c];
    const T E1 = U1[c] + K1[c];
    double delta = (double)(E0 - E1);
    if (isnan(delta)) delta = -INFINITY;
    const double pa = fmin(fmax(exp(delta), 0.0), 1.0);
    const bool acc = bern(u[c], pa);
    for (int j = lane; j < d; j += 32) {
        const i64 a = c * d + j;
        if (acc) p1[a] = -p1[a];
        else { q1[a] = q0[a]; p1[a] = p0[a]; g1[a] = g0[a]; }
    }
    if (lane == 0) {
        if (!acc) U1[c] = U0[c];
        p_accept[c] = pa;
        diverging[c] = fabs(delta) > thr ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------
// native draws exported in the injected layout
// ---------------------------------------------------------------------------
__global__ void philox_fill_kernel(RngView rng, i64 C, i64 T_, int d, int maxd, double* z, double* u_dir,
                                   double* u_biased, double* u_uniform, double* u_accept) {
    const i64 row = blockIdx.x;              // c*T + t
    const int c = (int)(row / T_), t = (int)(row % T_);
    const i64 nu = ((i64)1 << maxd) - 1;
    for (i64 k = threadIdx.x; k < d; k += blockDim.x) if (z) z[row * d + k] = draw_z(rng, c, t, (int)k, d);
    for (i64 k = threadIdx.x; k < maxd; k += blockDim.x) {
        if (u_dir) u_dir[row * maxd + k] = draw_u(rng, DRAW_DIR, c, t, (int)k, maxd);
        if (u_biased) u_biased[row * maxd + k] = draw_u(rng, DRAW_BIASED, c, t, (int)k, maxd);
    }
    if (u_uniform)
        for (i64 k = threadIdx.x; k < nu; k += blockDim.x)
            u_uniform[row * nu + k] = draw_u(rng, DRAW_UNIFORM, c, t, (int)k, maxd);
    if (u_accept && threadIdx.x == 0) u_accept[row] = draw_u(rng, DRAW_ACCEPT, c, t, 0, maxd);
}

// per-chain mean and variance over T draws [T][C][d] (split-R-hat / ESS building blocks)
template <typename T>
__global__ void chain_moments_kernel(const T* draws, i64 T_, i64 C, int d, double* mean, double* var) {
    i64 idx = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * d) return;
    double m = 0.0, m2 = 0.0;
    for (i64 t = 0; t < T_; ++t) {
        double x = (double)draws[t * C * d + idx];
        double dl = x - m;
        m += dl / (double)(t + 1);
        m2 += dl * (x - m);
    }
    mean[idx] = m;
    var[idx] = T_ > 1 ? m2 / (double)(T_ - 1) : 0.0;
}

// per-chain mean and biased autocovariance (divided by T, as Stan / arviz do) up to max_lag, by direct summation:
// one thread per (chain, dim, lag) -- diagnostics, not the hot path
template <typename T>
__global__ void chain_autocov_kernel(const T* draws, i64 T_, i64 C, int d, int max_lag, double* mean, double* acov) {
    const i64 cd = (i64)blockIdx.x;                  // chain * d + dim
    if (cd >= C * d) return;
    __shared__ double m_s;
    double part = 0.0;
    for (i64 t = threadIdx.x; t < T_; t += blockDim.x) part += (double)draws[t * C * d + cd];
    __shared__ double red[32];
    for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
        m_s = s / (double)T_;
        mean[cd] = m_s;
    }
    __syncthreads();
    const double m = m_s;
    for (int lag = threadIdx.x; lag <= max_lag; lag += blockDim.x) {
        double acc = 0.0;
        for (i64 t = 0; t + lag < T_; ++t)
            acc += ((double)draws[t * C * d + cd] - m) * ((double)draws[(t + lag) * C * d + cd] - m);
        acov[cd * (max_lag + 1) + lag] = acc / (double)T_;
    }
}

}  // namespace b2h

// ===========================================================================
// C-ABI
// ===========================================================================
using namespace b2h;

#define B2H_CHECK_CTX()                          \
    if (!ctx) {                                  \
        set_error("null context");               \
        return B2H_ERR_ARG;                      \
    }
#define B2H_TYPED(dtype, CALL_F32, CALL_F64)               \
    if ((dtype) == B2H_F64) { CALL_F64; }                  \
    else if ((dtype) == B2H_F32) { CALL_F32; }             \
    else { set_error("bad dtype"); return B2H_ERR_ARG; }

extern "C" {

int b2h_potential_and_grad(b2h_ctx* ctx, const b2h_model* model, int dtype, const void* q, void* U, void* g, int64_t C,
                           void* ws, int64_t ws_bytes) {
    B2H_CHECK_CTX();
    if (!model || !q || !U || !g || C <= 0) { set_error("bad argument"); return B2H_ERR_ARG; }
    B2H_TYPED(dtype, return potential_and_grad_impl<float>(ctx, model, (const float*)q, (float*)U, (float*)g, C, ws, ws_bytes),
              return potential_and_grad_impl<double>(ctx, model, (const double*)q, (double*)U, (double*)g, C, ws, ws_bytes));
}

int64_t b2h_potential_workspace_bytes(const b2h_model* model, int dtype, int64_t C) {
    return potential_workspace_bytes_impl(model, dtype, C);
}

int b2h_sample_momentum(b2h_ctx* ctx, const b2h_metric* metric, const b2h_rng* rng, int dtype, void* p, int64_t C,
                        int64_t d, int64_t transition, void* ws, int64_t ws_bytes) {
    B2H_CHECK_CTX();
    if (!metric || !rng || !p) { set_error("bad argument"); return B2H_ERR_ARG; }
    RngView rv;
    rv.mode = rng->mode; rv.key.k0 = (uint32_t)rng->seed; rv.key.k1 = (uint32_t)(rng->seed >> 32);
    rv.chain_offset = rng->chain_offset; rv.transition_offset = rng->transition_offset;
    rv.n_injected = rng->n_injected; rv.z = rng->z; rv.u_dir = rv.u_biased = rv.u_uniform = rv.u_accept = nullptr;
    ImmView iv = imm_view(metric, d);
    const bool dense = is_dense(metric);
    if (int rc = check_metric(metric, d)) return rc;
    const int tri = (metric->reserved & 1) ? 2 : 0;          // sqrt_t = L^-1 is lower-triangular
    const i64 n = C * d;
    const int eb = 256, eg = (int)((n + eb - 1) / eb);
    if (dense && (!ws || ws_bytes < n * (i64)dtype_size(dtype))) { set_error("momentum workspace too small"); return B2H_ERR_WORKSPACE; }
    cudaStream_t st = ctx->stream;
    if (dtype == B2H_F64) {
        momentum_kernel<double><<<eg, eb, 0, st>>>(iv, rv, dense ? (double*)ws : (double*)p, C, (int)d, (int)transition, dense);
        if (dense) metric_apply<double>(st, metric, (const double*)ws, metric->sqrt_t, (double*)p, C, (int)d, tri);
    } else if (dtype == B2H_F32) {
        momentum_kernel<float><<<eg, eb, 0, st>>>(iv, rv, dense ? (float*)ws : (float*)p, C, (int)d, (int)transition, dense);
        if (dense) metric_apply<float>(st, metric, (const float*)ws, metric->sqrt_t, (float*)p, C, (int)d, tri);
    } else { set_error("bad dtype"); return B2H_ERR_ARG; }
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_kinetic_energy(b2h_ctx* ctx, const b2h_metric* metric, int dtype, const void* p, void* K, int64_t C, int64_t d,
                       void* ws, int64_t ws_bytes) {
    B2H_CHECK_CTX();
    if (!metric || !p || !K) { set_error("bad argument"); return B2H_ERR_ARG; }
    ImmView iv = imm_view(metric, d);
    const bool dense = is_dense(metric);
    if (int rc = check_metric(metric, d)) return rc;
    if (dense && (!ws || ws_bytes < C * d * (i64)dtype_size(dtype))) { set_error("kinetic workspace too small"); return B2H_ERR_WORKSPACE; }
    cudaStream_t st = ctx->stream;
    const int grid = PGeo<32>::grid(C);
    if (dtype == B2H_F64) {
        if (dense) metric_apply<double>(st, metric, (const double*)p, metric->imm, (double*)ws, C, (int)d, 0);
        if (vec_ok(iv, d, dtype, {p, dense ? ws : nullptr})) kinetic_vec_kernel<double><<<grid, 128, 0, st>>>(iv, (const double*)p, dense ? (const double*)ws : nullptr, (double*)K, C, (int)d);
        else kinetic_kernel<double><<<grid, 128, 0, st>>>(iv, (const double*)p, dense ? (const double*)ws : nullptr, (double*)K, C, (int)d);
    } else if (dtype == B2H_F32) {
        if (dense) metric_apply<float>(st, metric, (const float*)p, metric->imm, (float*)ws, C, (int)d, 0);
        if (vec_ok(iv, d, dtype, {p, dense ? ws : nullptr})) kinetic_vec_kernel<float><<<grid, 128, 0, st>>>(iv, (const float*)p, dense ? (const float*)ws : nullptr, (float*)K, C, (int)d);
        else kinetic_kernel<float><<<grid, 128, 0, st>>>(iv, (const float*)p, dense ? (const float*)ws : nullptr, (float*)K, C, (int)d);
    } else { set_error("bad dtype"); return B2H_ERR_ARG; }
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_is_turning(b2h_ctx* ctx, const b2h_metric* metric, int dtype, const void* pl, const void* pr, const void* ps,
                   uint8_t* out, int64_t C, int64_t d, void* ws, int64_t ws_bytes) {
    B2H_CHECK_CTX();
    if (!metric || !pl || !pr || !ps || !out) { set_error("bad argument"); return B2H_ERR_ARG; }
    ImmView iv = imm_view(metric, d);
    const bool dense = is_dense(metric);
    if (int rc = check_metric(metric, d)) return rc;
    const i64 n = C * d;
    if (dense && (!ws || ws_bytes < 2 * n * (i64)dtype_size(dtype))) { set_error("is_turning workspace too small"); return B2H_ERR_WORKSPACE; }
    cudaStream_t st = ctx->stream;
    const int grid = PGeo<32>::grid(C);
    if (dtype == B2H_F64) {
        double* vl = dense ? (double*)ws : nullptr; double* vr = dense ? vl + n : nullptr;
        if (dense) {
            metric_apply<double>(st, metric, (const double*)pl, metric->imm, vl, C, (int)d, 0);
            metric_apply<double>(st, metric, (const double*)pr, metric->imm, vr, C, (int)d, 0);
        }
        if (vec_ok(iv, d, dtype, {pl, pr, ps, vl, vr})) turning_vec_kernel<double><<<grid, 128, 0, st>>>(iv, (const double*)pl, (const double*)pr, (const double*)ps, vl, vr, out, C, (int)d);
        else turning_kernel<double><<<grid, 128, 0, st>>>(iv, (const double*)pl, (const double*)pr, (const double*)ps, vl, vr, out, C, (int)d);
    } else if (dtype == B2H_F32) {
        float* vl = dense ? (float*)ws : nullptr; float* vr = dense ? vl + n : nullptr;
        if (dense) {
            metric_apply<float>(st, metric, (const float*)pl, metric->imm, vl, C, (int)d, 0);
            metric_apply<float>(st, metric, (const float*)pr, metric->imm, vr, C, (int)d, 0);
        }
        if (vec_ok(iv, d, dtype, {pl, pr, ps, vl, vr})) turning_vec_kernel<float><<<grid, 128, 0, st>>>(iv, (const float*)pl, (const float*)pr, (const float*)ps, vl, vr, out, C, (int)d);
        else turning_kernel<float><<<grid, 128, 0, st>>>(iv, (const float*)pl, (const float*)pr, (const float*)ps, vl, vr, out, C, (int)d);
    } else { set_error("bad dtype"); return B2H_ERR_ARG; }
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_leapfrog(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, int dtype, void* q, void* p, void* U,
                 void* g, const double* step_size, const int8_t* direction, int32_t n_steps, int64_t C, void* ws,
                 int64_t ws_bytes) {
    B2H_CHECK_CTX();
    if (!model || !metric || !q || !p || !U || !g || !step_size || n_steps < 0 || C <= 0) { set_error("bad argument"); return B2H_ERR_ARG; }
    B2H_TYPED(dtype,
              return leapfrog_typed<float>(ctx, model, metric, (float*)q, (float*)p, (float*)U, (float*)g, step_size, direction, n_steps, C, ws, ws_bytes),
              return leapfrog_typed<double>(ctx, model, metric, (double*)q, (double*)p, (double*)U, (double*)g, step_size, direction, n_steps, C, ws, ws_bytes));
}

int b2h_find_storage_indices(b2h_ctx* ctx, const int64_t* step, int64_t* imin, int64_t* imax, int64_t n) {
    B2H_CHECK_CTX();
    storage_indices_kernel<<<(int)((n + 255) / 256), 256, 0, ctx->stream>>>(step, imin, imax, n);
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_termination_update(b2h_ctx* ctx, int dtype, void* mck, void* sck, int64_t* imin, int64_t* imax, const void* msum,
                           const void* mom, const int64_t* step, int64_t C, int64_t d, int32_t maxd) {
    B2H_CHECK_CTX();
    const int grid = PGeo<32>::grid(C);
    ImmView none{};
    none.kind = B2H_IMM_SCALAR;
    if (vec_ok(none, d, dtype, {mck, sck, msum, mom})) {
        B2H_TYPED(dtype,
                  (termination_update_vec_kernel<float><<<grid, 128, 0, ctx->stream>>>((float*)mck, (float*)sck, imin, imax, (const float*)msum, (const float*)mom, step, C, (int)d, maxd)),
                  (termination_update_vec_kernel<double><<<grid, 128, 0, ctx->stream>>>((double*)mck, (double*)sck, imin, imax, (const double*)msum, (const double*)mom, step, C, (int)d, maxd)));
        B2H_LAUNCH_CHECK();
        return 0;
    }
    B2H_TYPED(dtype,
              (termination_update_kernel<float><<<grid, 128, 0, ctx->stream>>>((float*)mck, (float*)sck, imin, imax, (const float*)msum, (const float*)mom, step, C, (int)d, maxd)),
              (termination_update_kernel<double><<<grid, 128, 0, ctx->stream>>>((double*)mck, (double*)sck, imin, imax, (const double*)msum, (const double*)mom, step, C, (int)d, maxd)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_is_iterative_turning(b2h_ctx* ctx, const b2h_metric* metric, int dtype, const void* mck, const void* sck,
                             const int64_t* imin, const int64_t* imax, const void* msum, const void* mom, uint8_t* out,
                             int64_t C, int64_t d, int32_t maxd) {
    B2H_CHECK_CTX();
    if (is_dense(metric)) { set_error("is_iterative_turning primitive: dense metric not supported (use nuts_run)"); return B2H_ERR_UNSUPPORTED; }
    ImmView iv = imm_view(metric, d);
    const int grid = PGeo<32>::grid(C);
    if (vec_ok(iv, d, dtype, {mck, sck, msum, mom})) {
        B2H_TYPED(dtype,
                  (iterative_turning_vec_kernel<float><<<grid, 128, 0, ctx->stream>>>(iv, (const float*)mck, (const float*)sck, imin, imax, (const float*)msum, (const float*)mom, out, C, (int)d, maxd)),
                  (iterative_turning_vec_kernel<double><<<grid, 128, 0, ctx->stream>>>(iv, (const double*)mck, (const double*)sck, imin, imax, (const double*)msum, (const double*)mom, out, C, (int)d, maxd)));
        B2H_LAUNCH_CHECK();
        return 0;
    }
    B2H_TYPED(dtype,
              (iterative_turning_kernel<float><<<grid, 128, 0, ctx->stream>>>(iv, (const float*)mck, (const float*)sck, imin, imax, (const float*)msum, (const float*)mom, out, C, (int)d, maxd)),
              (iterative_turning_kernel<double><<<grid, 128, 0, ctx->stream>>>(iv, (const double*)mck, (const double*)sck, imin, imax, (const double*)msum, (const double*)mom, out, C, (int)d, maxd)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_dual_averaging_update(b2h_ctx* ctx, const double* p_accept, double target, double gamma, double t0, double kappa,
                              int64_t* step, double* x, double* x_avg, double* g_avg, const double* mu, int64_t C) {
    B2H_CHECK_CTX();
    dual_averaging_kernel<<<(int)((C + 255) / 256), 256, 0, ctx->stream>>>(p_accept, target, gamma, t0, kappa, step, x, x_avg, g_avg, mu, C);
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_welford_update(b2h_ctx* ctx, int dtype, const void* value, void* mean, void* m2, int64_t* n, int64_t C, int64_t d,
                       int32_t full) {
    B2H_CHECK_CTX();
    size_t smem = 2 * (size_t)d * dtype_size(dtype);
    if (smem > 48 * 1024) { set_error("welford: dim too large for the staging buffer"); return B2H_ERR_UNSUPPORTED; }
    B2H_TYPED(dtype,
              (welford_kernel<float><<<(int)C, 128, smem, ctx->stream>>>((const float*)value, (float*)mean, (float*)m2, n, C, (int)d, full)),
              (welford_kernel<double><<<(int)C, 128, smem, ctx->stream>>>((const double*)value, (double*)mean, (double*)m2, n, C, (int)d, full)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_mass_matrix_final(b2h_ctx* ctx, int dtype, const void* m2, const int64_t* n, void* out, int64_t C, int64_t d,
                          int32_t full) {
    B2H_CHECK_CTX();
    i64 total = C * (full ? d * d : d);
    int grid = (int)((total + 255) / 256);
    B2H_TYPED(dtype,
              (mass_matrix_final_kernel<float><<<grid, 256, 0, ctx->stream>>>((const float*)m2, n, (float*)out, C, (int)d, full)),
              (mass_matrix_final_kernel<double><<<grid, 256, 0, ctx->stream>>>((const double*)m2, n, (double*)out, C, (int)d, full)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_philox_fill(b2h_ctx* ctx, uint64_t seed, uint64_t chain_offset, uint64_t transition_offset, int64_t C,
                    int64_t n_transitions, int64_t d, int32_t maxd, double* z, double* u_dir, double* u_biased,
                    double* u_uniform, double* u_accept) {
    B2H_CHECK_CTX();
    RngView rv;
    memset(&rv, 0, sizeof(rv));
    rv.mode = 0; rv.key.k0 = (uint32_t)seed; rv.key.k1 = (uint32_t)(seed >> 32);
    rv.chain_offset = chain_offset; rv.transition_offset = transition_offset;
    philox_fill_kernel<<<(int)(C * n_transitions), 128, 0, ctx->stream>>>(rv, C, n_transitions, (int)d, maxd, z, u_dir, u_biased, u_uniform, u_accept);
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_dense_apply(b2h_ctx* ctx, int dtype, const void* in, const void* M, void* out, int64_t C, int64_t d) {
    B2H_CHECK_CTX();
    B2H_TYPED(dtype,
              launch_dense_apply<float>(ctx->stream, (const float*)in, (const float*)M, (float*)out, (int)C, (int)d, (int)d, nullptr, nullptr),
              launch_dense_apply<double>(ctx->stream, (const double*)in, (const double*)M, (double*)out, (int)C, (int)d, (int)d, nullptr, nullptr));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_chain_moments(b2h_ctx* ctx, int dtype, const void* draws, int64_t T_, int64_t C, int64_t d, double* mean,
                      double* var) {
    B2H_CHECK_CTX();
    int grid = (int)((C * d + 255) / 256);
    B2H_TYPED(dtype,
              (chain_moments_kernel<float><<<grid, 256, 0, ctx->stream>>>((const float*)draws, T_, C, (int)d, mean, var)),
              (chain_moments_kernel<double><<<grid, 256, 0, ctx->stream>>>((const double*)draws, T_, C, (int)d, mean, var)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_proposal_update(b2h_ctx* ctx, int dtype, const void* E0, const void* U, const void* K, double thr, void* energy,
                        double* weight, double* lpa, uint8_t* div, int64_t C) {
    B2H_CHECK_CTX();
    int grid = (int)((C + 255) / 256);
    B2H_TYPED(dtype,
              (proposal_update_kernel<float><<<grid, 256, 0, ctx->stream>>>((const float*)E0, (const float*)U, (const float*)K, thr, (float*)energy, weight, lpa, div, C)),
              (proposal_update_kernel<double><<<grid, 256, 0, ctx->stream>>>((const double*)E0, (const double*)U, (const double*)K, thr, (double*)energy, weight, lpa, div, C)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_progressive_sampling(b2h_ctx* ctx, int biased, const double* w_old, const double* w_new, const double* s_old,
                             const double* s_new, const double* u, uint8_t* acc, double* w_out, double* s_out, int64_t C) {
    B2H_CHECK_CTX();
    progressive_sampling_kernel<<<(int)((C + 255) / 256), 256, 0, ctx->stream>>>(biased, w_old, w_new, s_old, s_new, u, acc, w_out, s_out, C);
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_select_rows(b2h_ctx* ctx, int dtype, const uint8_t* mask, const void* a, const void* b, void* out, int64_t C,
                    int64_t d) {
    B2H_CHECK_CTX();
    int grid = (int)((C * d + 255) / 256);
    B2H_TYPED(dtype,
              (select_rows_kernel<float><<<grid, 256, 0, ctx->stream>>>(mask, (const float*)a, (const float*)b, (float*)out, C, (int)d)),
              (select_rows_kernel<double><<<grid, 256, 0, ctx->stream>>>(mask, (const double*)a, (const double*)b, (double*)out, C, (int)d)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_hmc_accept(b2h_ctx* ctx, int dtype, const b2h_state* old_state, b2h_state* new_state, const void* K_old,
                   const void* K_new, const double* u, double threshold, double* p_accept, uint8_t* is_diverging,
                   int64_t C, int64_t d) {
    B2H_CHECK_CTX();
    if (!old_state || !new_state || !K_old || !K_new || !u || !p_accept || !is_diverging) { set_error("null argument"); return B2H_ERR_ARG; }
    const int grid = (int)((C + 3) / 4);
    const b2h_state &o = *old_state, &n = *new_state;
    B2H_TYPED(dtype,
              (hmc_accept_kernel<float><<<grid, 128, 0, ctx->stream>>>((const float*)o.q, (const float*)o.p, (const float*)o.g, (const float*)o.U, (float*)n.q, (float*)n.p, (float*)n.g, (float*)n.U, (const float*)K_old, (const float*)K_new, u, threshold, p_accept, is_diverging, C, (int)d)),
              (hmc_accept_kernel<double><<<grid, 128, 0, ctx->stream>>>((const double*)o.q, (const double*)o.p, (const double*)o.g, (const double*)o.U, (double*)n.q, (double*)n.p, (double*)n.g, (double*)n.U, (const double*)K_old, (const double*)K_new, u, threshold, p_accept, is_diverging, C, (int)d)));
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_chain_autocov(b2h_ctx* ctx, int dtype, const void* draws, int64_t T_, int64_t C, int64_t d, int32_t max_lag,
                      double* mean, double* acov) {
    B2H_CHECK_CTX();
    if (!draws || !mean || !acov || T_ < 2 || max_lag < 0 || max_lag >= T_) { set_error("bad argument"); return B2H_ERR_ARG; }
    int grid = (int)(C * d);
    B2H_TYPED(dtype,
              (chain_autocov_kernel<float><<<grid, 128, 0, ctx->stream>>>((const float*)draws, T_, C, (int)d, max_lag, mean, acov)),
              (chain_autocov_kernel<double><<<grid, 128, 0, ctx->stream>>>((const double*)draws, T_, C, (int)d, max_lag, mean, acov)));
    B2H_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
