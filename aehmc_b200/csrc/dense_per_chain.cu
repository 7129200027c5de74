// Per-chain dense inverse mass matrices (B2H_IMM_DENSE_PER_CHAIN): chain c has its own imm[c], sqrt_t[c] and
// chol_t[c], [d x d] row-major at c * d * d.
//
//  - pc_apply_kernel: the batched per-chain row-vector x matrix product out[r] = in[r] . M[chain(r)].  It serves the
//    dense metric's mat-vecs (w' = imm . g' of every tick, the primitives) and, with a device-side row count and a
//    row -> chain list, the momentum rider of the split engine (p0 = z . sqrt_t and v0 = z . chol_t from one read of
//    the compact normals z).  Memory-bound: every matrix element is read once and used in one FMA.
//  - pc_factor_kernel: symmetrisation, Cholesky and triangular inverse of every chain's matrix, one CTA per chain,
//    the matrix in shared memory as FP64.  Runs once per metric construction / window end.
//
// Every output element is a sum over k in ascending order with no reassociation, so integer inputs give the exact
// product and the result does not depend on the launch geometry.
#include <algorithm>

#include "common.cuh"
#include "launch.h"

namespace b2h {

constexpr int kPcThreads = 256;
constexpr int kPcMaxBlocks = 4096;     // grid-stride beyond this (the rider's grid is sized for C rows, most idle)

template <typename T> struct PcVec;
template <> struct PcVec<double> { static constexpr int N = 2; using type = double2; };
template <> struct PcVec<float> { static constexpr int N = 4; using type = float4; };

// tri: 0 full; 1 M upper-triangular (M[k][j] = 0 for k > j); 2 lower-triangular (M[k][j] = 0 for k < j).  The zero
// half is never used, whatever it holds.
B2H_DEVINL bool pc_used(int tri, int k, int j) { return tri == 0 || (tri == 1 ? k <= j : k >= j); }

template <typename T, int VEC>
B2H_DEVINL void pc_load(T (&v)[VEC], const T* p) {
    if constexpr (VEC == 1) {
        v[0] = __ldg(p);
    } else {
        typename PcVec<T>::type x = __ldg((const typename PcVec<T>::type*)p);
        const T* e = (const T*)&x;
#pragma unroll
        for (int i = 0; i < VEC; ++i) v[i] = e[i];
    }
}

template <typename T, int VEC>
B2H_DEVINL void pc_store(T* p, const T (&v)[VEC]) {
    if constexpr (VEC == 1) {
        p[0] = v[0];
    } else {
        typename PcVec<T>::type x;
        T* e = (T*)&x;
#pragma unroll
        for (int i = 0; i < VEC; ++i) e[i] = v[i];
        *(typename PcVec<T>::type*)p = x;
    }
}

// A CTA holds cpb = kPcThreads / tpc rows; the tpc threads of a row own VEC adjacent output columns each.  The rows'
// inputs are staged in shared memory (every thread of a row reads all d of them).
template <typename T, int VEC, int NM>
__global__ void __launch_bounds__(kPcThreads) pc_apply_kernel(PcJob<T> a, int tpc) {
    extern __shared__ unsigned char pc_smem[];
    T* zin = (T*)pc_smem;
    const int d = a.d, cpb = kPcThreads / tpc;
    const int slot = threadIdx.x / tpc, lane = threadIdx.x % tpc;
    const i64 n = a.count ? min((i64)*a.count, a.rows) : a.rows;
    const i64 dd = (i64)d * d;
    for (i64 r0 = (i64)blockIdx.x * cpb; r0 < n; r0 += (i64)gridDim.x * cpb) {
        __syncthreads();
        const i64 lim = min((i64)cpb, n - r0) * d;
        for (int i = threadIdx.x; i < cpb * d; i += kPcThreads) zin[i] = i < lim ? a.in[r0 * d + i] : (T)0;
        __syncthreads();
        const i64 r = r0 + slot;
        if (r >= n) continue;
        const i64 c = a.list ? (i64)a.list[r] : r;
        const T* x = zin + slot * d;
        for (int j0 = lane * VEC; j0 < d; j0 += tpc * VEC) {
            T acc[NM][VEC];
#pragma unroll
            for (int m = 0; m < NM; ++m)
#pragma unroll
                for (int i = 0; i < VEC; ++i) acc[m][i] = 0;
            // k range touching any of the VEC columns: upper -> [0, j0 + VEC), lower -> [j0, d)
            int klo = 0, khi = d;
            if (NM == 1 && a.tri[0] == 1) khi = min(d, j0 + VEC);
            if (NM == 1 && a.tri[0] == 2) klo = j0;
#pragma unroll 4
            for (int k = klo; k < khi; ++k) {
                const T xk = x[k];
#pragma unroll
                for (int m = 0; m < NM; ++m) {
                    const int tri = a.tri[m];
                    if (NM > 1 && !(tri == 0 || (tri == 1 ? k < j0 + VEC : k >= j0))) continue;
                    T mv[VEC];
                    pc_load<T, VEC>(mv, a.M[m] + c * dd + (i64)k * d + j0);
#pragma unroll
                    for (int i = 0; i < VEC; ++i)
                        if (pc_used(tri, k, j0 + i)) acc[m][i] = fma(xk, mv[i], acc[m][i]);
                }
            }
#pragma unroll
            for (int m = 0; m < NM; ++m) pc_store<T, VEC>(a.out[m] + c * d + j0, acc[m]);
        }
    }
}

// The one place that decides between the 128-bit and the scalar path: every row of every matrix and of the output
// starts 16-byte aligned iff d is a multiple of VEC and the base pointers are 16-byte aligned.  The inputs go through
// shared memory element by element and need no alignment.
template <typename T>
static bool pc_vector_layout(const PcJob<T>& a, int nm) {
    if (a.d % PcVec<T>::N) return false;
    for (int m = 0; m < nm; ++m)
        if (((uintptr_t)a.M[m] & 15) || ((uintptr_t)a.out[m] & 15)) return false;
    return true;
}

template <typename T, int VEC, int NM>
static void pc_launch(cudaStream_t st, const PcJob<T>& a) {
    const int groups = (a.d + VEC - 1) / VEC;
    int tpc = 1;
    while (tpc < groups && tpc < kPcThreads) tpc <<= 1;
    const int cpb = kPcThreads / tpc;
    const i64 blocks = std::min<i64>((a.rows + cpb - 1) / cpb, kPcMaxBlocks);
    pc_apply_kernel<T, VEC, NM><<<(int)blocks, kPcThreads, (size_t)cpb * a.d * sizeof(T), st>>>(a, tpc);
}

template <typename T>
void launch_dense_pc(cudaStream_t st, const PcJob<T>& a) {
    if (a.rows <= 0) return;
    const int nm = a.M[1] ? 2 : 1;
    const bool vec = pc_vector_layout<T>(a, nm);
    constexpr int V = PcVec<T>::N;
    if (nm == 2) {
        if (vec) pc_launch<T, V, 2>(st, a);
        else pc_launch<T, 1, 2>(st, a);
    } else {
        if (vec) pc_launch<T, V, 1>(st, a);
        else pc_launch<T, 1, 1>(st, a);
    }
}

template <typename T>
void launch_dense_apply_pc(cudaStream_t st, const T* in, const T* M, T* out, i64 C, int d, int tri) {
    PcJob<T> a{in, {M, nullptr}, {out, nullptr}, {tri, 0}, nullptr, nullptr, C, d};
    launch_dense_pc<T>(st, a);
}

template void launch_dense_pc<float>(cudaStream_t, const PcJob<float>&);
template void launch_dense_pc<double>(cudaStream_t, const PcJob<double>&);
template void launch_dense_apply_pc<float>(cudaStream_t, const float*, const float*, float*, i64, int, int);
template void launch_dense_apply_pc<double>(cudaStream_t, const double*, const double*, double*, i64, int, int);

// One CTA per chain.  a = (A + A^T) / 2 in FP64 shared memory; right-looking Cholesky overwrites its lower triangle
// with L; then thread j solves L x = e_j by forward substitution (fixed ascending order) and keeps X = L^-1 transposed
// in the strict upper triangle (X[i][j] at a[j][i], i > j) and its diagonal in xd.  A pivot that is not positive
// (or NaN) stops the chain: info = k + 1 and every output of the chain is NaN.
template <typename T>
__global__ void __launch_bounds__(256) pc_factor_kernel(const T* imm_in, T* imm, T* sqrt_t, T* chol_t, int* info, int d) {
    extern __shared__ double pf_smem[];
    double* a = pf_smem;
    double* xd = a + (size_t)d * d;
    __shared__ int fail;
    const int tid = threadIdx.x, bs = blockDim.x;
    const i64 dd = (i64)d * d, base = (i64)blockIdx.x * dd;
    for (int idx = tid; idx < d * d; idx += bs) {
        const int i = idx / d, j = idx % d;
        a[idx] = 0.5 * ((double)imm_in[base + (i64)i * d + j] + (double)imm_in[base + (i64)j * d + i]);
    }
    if (tid == 0) fail = 0;
    __syncthreads();                                  // imm_in is fully read: imm may alias it
    for (int idx = tid; idx < d * d; idx += bs) imm[base + idx] = (T)a[idx];
    for (int k = 0; k < d; ++k) {
        const double piv = a[k * d + k];
        if (!(piv > 0.0)) {
            if (tid == 0) fail = k + 1;
            break;                                    // uniform: every thread read the same pivot
        }
        const double lkk = sqrt(piv);
        __syncthreads();
        if (tid == 0) a[k * d + k] = lkk;
        for (int i = k + 1 + tid; i < d; i += bs) a[i * d + k] = a[i * d + k] / lkk;
        __syncthreads();
        const int m = d - k - 1;
        for (int idx = tid; idx < m * m; idx += bs) {
            const int i = k + 1 + idx / m, j = k + 1 + idx % m;
            if (j <= i) a[i * d + j] = fma(-a[i * d + k], a[j * d + k], a[i * d + j]);
        }
        __syncthreads();
    }
    __syncthreads();
    const bool ok = fail == 0;
    if (ok) {
        for (int j = tid; j < d; j += bs) {
            const double xjj = 1.0 / a[j * d + j];
            xd[j] = xjj;
            for (int i = j + 1; i < d; ++i) {
                double s = a[i * d + j] * xjj;                                      // L[i][j] X[j][j]
                for (int k = j + 1; k < i; ++k) s = fma(a[i * d + k], a[j * d + k], s);   // L[i][k] X[k][j]
                a[j * d + i] = -s / a[i * d + i];
            }
        }
    }
    __syncthreads();
    const T nan = (T)NAN;
    for (int idx = tid; idx < d * d; idx += bs) {
        const int i = idx / d, j = idx % d;
        if (!ok) {
            imm[base + idx] = nan; sqrt_t[base + idx] = nan; chol_t[base + idx] = nan;
            continue;
        }
        // sqrt_t = X = L^-1 (lower), chol_t = L^T (upper)
        sqrt_t[base + idx] = (T)(i > j ? a[j * d + i] : (i == j ? xd[i] : 0.0));
        chol_t[base + idx] = (T)(j > i ? a[j * d + i] : (i == j ? a[i * d + i] : 0.0));
    }
    if (tid == 0) info[blockIdx.x] = fail;
}

template <typename T>
static int factor_typed(b2h_ctx* ctx, const T* in, T* imm, T* sqrt_t, T* chol_t, int* info, i64 C, int d) {
    const size_t smem = ((size_t)d * d + d) * sizeof(double);
    B2H_CUDA(cudaFuncSetAttribute(pc_factor_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pc_factor_kernel<T><<<(unsigned)C, 256, smem, ctx->stream>>>(in, imm, sqrt_t, chol_t, info, d);
    B2H_LAUNCH_CHECK();
    return 0;
}

}  // namespace b2h

using namespace b2h;

extern "C" {

int b2h_dense_apply_per_chain(b2h_ctx* ctx, int dtype, const void* in, const void* M, void* out, int64_t C, int64_t d,
                              int32_t tri) {
    if (!ctx) { set_error("null context"); return B2H_ERR_ARG; }
    if (!in || !M || !out) { set_error("null argument"); return B2H_ERR_ARG; }
    if (C < 1 || C > (1ll << 30)) { set_error("dense_apply_per_chain: C must be in [1, 2^30]"); return B2H_ERR_ARG; }
    if (d < 1 || d > B2H_DENSE_PER_CHAIN_MAX_DIM) {
        set_error("dense_apply_per_chain: d must be in [1, B2H_DENSE_PER_CHAIN_MAX_DIM]");
        return B2H_ERR_ARG;
    }
    if (tri < 0 || tri > 2) { set_error("dense_apply_per_chain: tri must be 0, 1 or 2"); return B2H_ERR_ARG; }
    if (dtype == B2H_F64) launch_dense_apply_pc<double>(ctx->stream, (const double*)in, (const double*)M, (double*)out, C, (int)d, tri);
    else if (dtype == B2H_F32) launch_dense_apply_pc<float>(ctx->stream, (const float*)in, (const float*)M, (float*)out, C, (int)d, tri);
    else { set_error("bad dtype"); return B2H_ERR_ARG; }
    B2H_LAUNCH_CHECK();
    return 0;
}

int b2h_dense_factor_per_chain(b2h_ctx* ctx, int dtype, const void* imm_in, void* imm, void* sqrt_t, void* chol_t,
                               int32_t* info, int64_t C, int64_t d) {
    if (!ctx) { set_error("null context"); return B2H_ERR_ARG; }
    if (!imm_in || !imm || !sqrt_t || !chol_t || !info) { set_error("null argument"); return B2H_ERR_ARG; }
    if (C < 1 || C > (1ll << 30)) { set_error("dense_factor_per_chain: C must be in [1, 2^30]"); return B2H_ERR_ARG; }
    if (d < 1 || d > B2H_DENSE_PER_CHAIN_MAX_DIM) {
        set_error("dense_factor_per_chain: d must be in [1, B2H_DENSE_PER_CHAIN_MAX_DIM]");
        return B2H_ERR_ARG;
    }
    if (dtype == B2H_F64)
        return factor_typed<double>(ctx, (const double*)imm_in, (double*)imm, (double*)sqrt_t, (double*)chol_t, info, C, (int)d);
    if (dtype == B2H_F32)
        return factor_typed<float>(ctx, (const float*)imm_in, (float*)imm, (float*)sqrt_t, (float*)chol_t, info, C, (int)d);
    set_error("bad dtype");
    return B2H_ERR_ARG;
}

}  // extern "C"
