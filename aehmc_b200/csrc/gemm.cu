// Dense apply for all chains at once:  out[M x N] = A[M x K] . B[K x N]
//
// This is the mass-matrix apply (metrics.py:71,95-96: velocity = imm @ p) and the
// correlated-Gaussian gradient (Lambda (q - mu)) of every chain in one launch.
// B is shared by all chains, so the per-chain mat-vecs of the reference become
// one [C x d].[d x d] product: FP64/FP32 FMA-pipe bound, not HBM bound
// (SURVEY.md section 8d).  FP64 has no tcgen05 path on sm_100a, so this is a
// register-tiled SIMT kernel: 128x128x16 CTA tile, 256 threads, 8x8 outputs per
// thread laid out as 4x4 chunks of 2 so that every shared-memory read is a
// conflict-free 128-bit load; global->shared is software-pipelined through
// registers and the shared->register fragments are double-buffered.
//
// One launch can carry TWO problems ("groups") that share N and K: the engine
// uses the second group for the few momentum rows of chains that start a new
// transition (p0 = z . sqrt^T, v0 = p0 . imm), whose row count is only known on
// the device and which would otherwise cost a full launch latency each.  Rows
// can be gathered (in_rows) and scattered (out_rows) through index lists.
#include <algorithm>
#include <climits>
#include <type_traits>
#include <stdlib.h>

#include "common.cuh"
#include "launch.h"

namespace b2h {

constexpr int BM = 128, BN = 128, BK = 16, GT = 256;

template <typename T>
__global__ void __launch_bounds__(GT, 1)
dense_apply_kernel(GemmGroup<T> g0, GemmGroup<T> g1, GemmGroup<T> g2, int N, int K, int tiles_n, int tiles_m0,
                   int tiles_m1, int k_chunk, i64 split_stride) {
    int tile_m = blockIdx.x / tiles_n;
    const int tile_n = blockIdx.x % tiles_n;
    const int which = tile_m < tiles_m0 ? 0 : (tile_m < tiles_m0 + tiles_m1 ? 1 : 2);
    const GemmGroup<T>& g = which == 0 ? g0 : (which == 1 ? g1 : g2);
    tile_m -= which == 0 ? 0 : (which == 1 ? tiles_m0 : tiles_m0 + tiles_m1);
    int M = g.M;
    if (g.m_dev) M = min(M, *g.m_dev);
    const int m0 = tile_m * BM, n0 = tile_n * BN;
    if (m0 >= M) return;
    const T* __restrict__ A = g.A;
    const T* __restrict__ B = g.B;
    const T* __restrict__ sub = g.sub;
    const i64 lda = g.lda, ldb = g.ldb, ldo = g.ldo;
    // split-K: slice blockIdx.y handles k in [k_begin, k_end) and writes its own partial plane
    const int k_begin = blockIdx.y * k_chunk;
    const int k_end = min(K, k_begin + k_chunk);
    T* __restrict__ out = g.out + (i64)blockIdx.y * split_stride;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef T (*TileA)[BK][BM];
    typedef T (*TileB)[BK][BN];
    TileA As = reinterpret_cast<TileA>(smem_raw);                                  // [2][k][m] (transposed)
    TileB Bs = reinterpret_cast<TileB>(smem_raw + 2 * BK * BM * sizeof(T));        // [2][k][n]

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;

    // global->smem assignment.  A tile 128 rows x 16 k: a warp takes 32 consecutive rows, each thread 8
    // consecutive k of its row (two full 32-byte sectors); the transposed smem stores are conflict-free.
    const int a_row = tid & 127, a_k = (tid >> 7) * 8;
    // B tile 16 k x 128 n: a warp reads 512 contiguous bytes of one k row (2 n per thread), 4 k rows per thread.
    const int b_k = tid >> 6, b_n = (tid & 63) * 2;

    i64 a_src = -1;
    {
        const int gr = m0 + a_row;
        if (gr < M) a_src = (i64)(g.in_rows ? g.in_rows[gr] : gr) * lda;
    }

    T acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = (T)0;

    T ra[8], rb[8];
    auto load_tile = [&](int k0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int gk = k0 + a_k + i;
            T x = (T)0;
            if (a_src >= 0 && gk < k_end) {
                x = A[a_src + gk];
                if (sub) x -= sub[gk];
            }
            ra[i] = x;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int gk = k0 + b_k + 4 * i, gn = n0 + b_n;
            rb[2 * i] = (gk < k_end && gn < N) ? B[(i64)gk * ldb + gn] : (T)0;
            rb[2 * i + 1] = (gk < k_end && gn + 1 < N) ? B[(i64)gk * ldb + gn + 1] : (T)0;
        }
    };
    auto store_tile = [&](int buf) {
#pragma unroll
        for (int i = 0; i < 8; ++i) As[buf][a_k + i][a_row] = ra[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            Bs[buf][b_k + 4 * i][b_n] = rb[2 * i];
            Bs[buf][b_k + 4 * i][b_n + 1] = rb[2 * i + 1];
        }
    };
    auto load_frag = [&](int buf, int kk, T (&a)[8], T (&b)[8]) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            // rows ty*2 + 32*c + {0,1}, cols tx*2 + 32*c + {0,1}
            a[2 * c] = As[buf][kk][ty * 2 + 32 * c];
            a[2 * c + 1] = As[buf][kk][ty * 2 + 32 * c + 1];
            b[2 * c] = Bs[buf][kk][tx * 2 + 32 * c];
            b[2 * c + 1] = Bs[buf][kk][tx * 2 + 32 * c + 1];
        }
    };

    const int nk = (k_end - k_begin + BK - 1) / BK;
    load_tile(k_begin);
    store_tile(0);
    __syncthreads();
    T fa[2][8], fb[2][8];
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) load_tile(k_begin + (kt + 1) * BK);
        load_frag(buf, 0, fa[0], fb[0]);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const int cur = kk & 1;
            if (kk + 1 < BK) load_frag(buf, kk + 1, fa[cur ^ 1], fb[cur ^ 1]);
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fma(fa[cur][i], fb[cur][j], acc[i][j]);
        }
        if (kt + 1 < nk) {
            store_tile(buf ^ 1);
            __syncthreads();
        }
    }

#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int gr = m0 + ty * 2 + 32 * (i >> 1) + (i & 1);
        if (gr >= M) continue;
        const i64 orow = (i64)(g.out_rows ? g.out_rows[gr] : gr) * ldo;
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            const int gn = n0 + tx * 2 + 32 * (j >> 1);
            if (gn + 1 < N) {
                out[orow + gn] = acc[i][j];
                out[orow + gn + 1] = acc[i][j + 1];
            } else if (gn < N) {
                out[orow + gn] = acc[i][j];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// FP64: same CTA tile, but the inner product runs on the FP64 tensor path (mma.sync m8n8k4, SASS DMMA --
// the only tensor-core path FP64 has on sm_100a; tcgen05 has no f64 kind).  8 warps as 4 (M) x 2 (N),
// warp tile 32 x 64 = 4 x 8 DMMA tiles, 64 accumulators per thread.  Versus the FMA-pipe version this
// needs 8x fewer issue slots and ~5x fewer shared-memory loads per FMA.  Shared rows are padded to 136
// doubles so that the 4 k-rows x 8 columns a warp reads per fragment land in 2 wavefronts (the minimum).
// ---------------------------------------------------------------------------------------------
constexpr int DPAD = 8, DLD = BM + DPAD;

// D(16x8) += A(16xKI) . B(KIx8), FP64.  Fragment ownership (lane = 4*g + t): a[2i] = A[g][t+4i],
// a[2i+1] = A[g+8][t+4i]; b[i] = B[t+4i][g]; c0,c1 = C[g][2t..2t+1], c2,c3 = C[g+8][2t..2t+1].
template <int KI> struct Dmma;
template <> struct Dmma<4> {
    __device__ __forceinline__ static void run(double (&c)[4], const double* a, const double* b) {
        asm volatile("mma.sync.aligned.m16n8k4.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                     : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3]) : "d"(a[0]), "d"(a[1]), "d"(b[0]));
    }
};
template <> struct Dmma<8> {
    __device__ __forceinline__ static void run(double (&c)[4], const double* a, const double* b) {
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
                     : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(b[0]), "d"(b[1]));
    }
};
template <> struct Dmma<16> {
    __device__ __forceinline__ static void run(double (&c)[4], const double* a, const double* b) {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
                     "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
                     : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
                     : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(a[4]), "d"(a[5]), "d"(a[6]), "d"(a[7]),
                       "d"(b[0]), "d"(b[1]), "d"(b[2]), "d"(b[3]));
    }
};

template <int KI>
__global__ void __launch_bounds__(GT, 1)
dense_apply_dmma_kernel(GemmGroup<double> g0, GemmGroup<double> g1, GemmGroup<double> g2, int N, int K, int tiles_n,
                        int tiles_m0, int tiles_m1, int k_chunk, i64 split_stride) {
    typedef double T;
    int tile_m = blockIdx.x / tiles_n;
    const int tile_n = blockIdx.x % tiles_n;
    const int which = tile_m < tiles_m0 ? 0 : (tile_m < tiles_m0 + tiles_m1 ? 1 : 2);
    const GemmGroup<T>& g = which == 0 ? g0 : (which == 1 ? g1 : g2);
    tile_m -= which == 0 ? 0 : (which == 1 ? tiles_m0 : tiles_m0 + tiles_m1);
    int M = g.M;
    if (g.m_dev) M = min(M, *g.m_dev);
    const int m0 = tile_m * BM, n0 = tile_n * BN;
    if (m0 >= M) return;
    const T* __restrict__ A = g.A;
    const T* __restrict__ B = g.B;
    const T* __restrict__ sub = g.sub;
    const i64 lda = g.lda, ldb = g.ldb, ldo = g.ldo;
    const int k_begin = blockIdx.y * k_chunk;
    const int k_end = min(K, k_begin + k_chunk);
    T* __restrict__ out = g.out + (i64)blockIdx.y * split_stride;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* As = reinterpret_cast<T*>(smem_raw);                       // [2][BK][DLD]  (k-major: A transposed)
    T* Bs = As + 2 * BK * DLD;                                    // [2][BK][DLD]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 64;        // warp tile origin inside the CTA tile
    const int gq = lane >> 2, tq = lane & 3;                      // MMA fragment coordinates

    const int a_row = tid & 127, a_k = (tid >> 7) * 8;
    const int b_k = tid >> 6, b_n = (tid & 63) * 2;
    i64 a_src = -1;
    {
        const int gr = m0 + a_row;
        if (gr < M) a_src = (i64)(g.in_rows ? g.in_rows[gr] : gr) * lda;
    }

    T acc[2][8][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.0;

    T ra[8], rb[8];
    auto load_tile = [&](int k0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int gk = k0 + a_k + i;
            T x = 0.0;
            if (a_src >= 0 && gk < k_end) {
                x = A[a_src + gk];
                if (sub) x -= sub[gk];
            }
            ra[i] = x;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int gk = k0 + b_k + 4 * i, gn = n0 + b_n;
            rb[2 * i] = (gk < k_end && gn < N) ? B[(i64)gk * ldb + gn] : 0.0;
            rb[2 * i + 1] = (gk < k_end && gn + 1 < N) ? B[(i64)gk * ldb + gn + 1] : 0.0;
        }
    };
    auto store_tile = [&](int buf) {
        T* as = As + buf * BK * DLD;
        T* bs = Bs + buf * BK * DLD;
#pragma unroll
        for (int i = 0; i < 8; ++i) as[(a_k + i) * DLD + a_row] = ra[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            bs[(b_k + 4 * i) * DLD + b_n] = rb[2 * i];
            bs[(b_k + 4 * i) * DLD + b_n + 1] = rb[2 * i + 1];
        }
    };

    const int nk = (k_end - k_begin + BK - 1) / BK;
    load_tile(k_begin);
    store_tile(0);
    __syncthreads();
    constexpr int NI = KI / 4;                                    // k-quads per instruction
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) load_tile(k_begin + (kt + 1) * BK);
        const T* as = As + buf * BK * DLD + wm + gq;
        const T* bs = Bs + buf * BK * DLD + wn + gq;
#pragma unroll
        for (int k0 = 0; k0 < BK; k0 += KI) {
            T fa[2][2 * NI], fb[8][NI];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int q = 0; q < NI; ++q) {
                    fa[i][2 * q] = as[(k0 + tq + 4 * q) * DLD + i * 16];
                    fa[i][2 * q + 1] = as[(k0 + tq + 4 * q) * DLD + i * 16 + 8];
                }
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int q = 0; q < NI; ++q) fb[j][q] = bs[(k0 + tq + 4 * q) * DLD + j * 8];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) Dmma<KI>::run(acc[i][j], fa[i], fb[j]);
        }
        if (kt + 1 < nk) {
            store_tile(buf ^ 1);
            __syncthreads();
        }
    }

#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int gr = m0 + wm + i * 16 + h * 8 + gq;
            if (gr >= M) continue;
            const i64 orow = (i64)(g.out_rows ? g.out_rows[gr] : gr) * ldo;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int gn = n0 + wn + j * 8 + tq * 2;
                if (gn + 1 < N) {
                    out[orow + gn] = acc[i][j][2 * h];
                    out[orow + gn + 1] = acc[i][j][2 * h + 1];
                } else if (gn < N) {
                    out[orow + gn] = acc[i][j][2 * h];
                }
            }
        }
}

// ---------------------------------------------------------------------------------------------
// FP64 main path: the same DMMA warp tiling fed by a 3-stage cp.async (LDGSTS) pipeline -- no register
// staging, one barrier per k-tile -- and a CTA tile width chosen per problem (BN = 128 / 112 / 96) so
// that the tile count fills whole waves of 148 SMs (d = 1000: 32 x 9 tiles of 128 x 112 = 288 of 296
// slots).  A stays row-major [m][k] in shared memory, B is [k][n]; row paddings: see kApad / kBpad below.  The two
// warps of a scheduler refill the freed stage at different points of a k-tile, launches without a vector to subtract
// take a loop body without the subtraction, launches whose row count lives on the device walk the valid tiles with a
// small grid (LOOP).
// Requires 16-byte aligned rows (even K, N, leading dimensions); otherwise the register-staged kernel runs.
// ---------------------------------------------------------------------------------------------
constexpr int STAGES = 3;
#ifndef B2H_GEMM_WARPS_DEFAULT
#define B2H_GEMM_WARPS_DEFAULT 8
#endif
#ifndef B2H_GEMM_BK_DEFAULT
#define B2H_GEMM_BK_DEFAULT 32
#endif

// Fragment loads: every lane fetches TWO fragment values per shared-memory load (LDS.128) -- the k-slots tq / tq + 4 of
// the m16n8k8 shape are bound to the adjacent reduction indices 2 tq / 2 tq + 1 (the same binding for A and B, so the
// product is unchanged up to the order of the partial sums) and the n8 tiles 2 p / 2 p + 1 of a warp take the even / odd
// columns of a 16-column group.  12 loads per 14 MMAs instead of the 22 of one value per load; the paddings make the
// quarter-warp accesses conflict free (A rows shift by 16 banks, B row pairs by 8).
constexpr int kApad = 8;
constexpr int kBpad = 2;

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(d), "l"(gsrc), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async16s(unsigned sdst, const void* gsrc, int src_bytes) {   // shared-space address
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(sdst), "l"(gsrc), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async16p(unsigned sdst, const void* gsrc, int src_bytes, bool active) {   // predicated
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %3, 0;\n\t@p cp.async.cg.shared.global [%0], [%1], 16, %2;\n\t}"
                 :: "r"(sdst), "l"(gsrc), "r"(src_bytes), "r"((int)active));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N_> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N_)); }

// MI: 16-row MMA tiles per warp along M.  MI = 2: 8 warps (4 x 2), warp tile 32 x BN_/2.  MI = 1: 16 warps (8 x 2), warp
// tile 16 x BN_/2 -- half the accumulators per thread, twice the warps to cover the per-k-tile barrier.
// BK_: k-tile depth (16, or 32: half the barriers and commit groups per flop, 203 KB of shared memory for 3 stages).
template <int BN_, int MI, int BK_, bool LOOP>
__global__ void __launch_bounds__((128 / (16 * MI)) * 2 * 32, 1)
dense_apply_dmma_async_kernel(GemmGroup<double> g0, GemmGroup<double> g1, GemmGroup<double> g2, int N, int K, int tiles_n,
                              int tiles_m0, int tiles_m1, int k_chunk_in, i64 split_stride, int total_tiles) {
    typedef double T;
    constexpr int NJ = BN_ / 16;               // 8-wide MMA tiles per warp along N (warp tile 16 MI x BN_/2)
    constexpr int WROWS = 128 / (16 * MI);     // warps along M
    constexpr int NT = WROWS * 2 * 32;         // threads of the CTA
    constexpr int ALD_ = BK_ + kApad;          // padded A row (doubles)
    constexpr int CPR = BK_ / 2;               // 16-byte chunks per A row
    constexpr int A_ITERS = (BM * CPR) / NT;   // 16-byte chunks of the A tile per thread
    constexpr int BLD = BN_ + kBpad;
    constexpr int A_STAGE = BM * ALD_, B_STAGE = BK_ * BLD;
    // One tile per CTA (gridDim.x == total_tiles), except for launches whose row count only the device knows (the
    // momentum contractions of restarting chains: the grid would cover all C rows and 9 of 10 CTAs -- each needing a
    // whole SM's shared memory -- would exit at once): a small grid walks the tiles and skips the empty ones.
    // LOOP: the walk enumerates only the row tiles that hold rows (vt0 / vt1 / vt2 of the three groups, from the
    // device-side counts), so that the few valid tiles spread evenly over the grid
    int vt0 = tiles_m0, vt1 = tiles_m1, vt2 = total_tiles / tiles_n - tiles_m0 - tiles_m1;
    if (LOOP) {
        if (g0.m_dev) vt0 = min(vt0, (min(g0.M, *g0.m_dev) + BM - 1) / BM);
        if (g1.m_dev) vt1 = min(vt1, (min(g1.M, *g1.m_dev) + BM - 1) / BM);
        if (g2.m_dev) vt2 = min(vt2, (min(g2.M, *g2.m_dev) + BM - 1) / BM);
        total_tiles = (vt0 + vt1 + vt2) * tiles_n;
        if ((int)blockIdx.x >= total_tiles) return;
    }
    int tile = blockIdx.x;
    do {
    if (LOOP && tile != (int)blockIdx.x) __syncthreads();         // every warp is done with the previous tile's stages
    int k_chunk = k_chunk_in;
    int tile_m = tile / tiles_n;
    const int tile_n = tile % tiles_n;
    const int which = tile_m < vt0 ? 0 : (tile_m < vt0 + vt1 ? 1 : 2);
    const GemmGroup<T>& g = which == 0 ? g0 : (which == 1 ? g1 : g2);
    tile_m -= which == 0 ? 0 : (which == 1 ? vt0 : vt0 + vt1);
    int M = g.M;
    if (g.m_dev) M = min(M, *g.m_dev);
    const int m0 = tile_m * BM, n0 = tile_n * BN_;
    if (m0 >= M) continue;
    const T* __restrict__ A = g.A;
    const T* __restrict__ B = g.B;
    const T* __restrict__ sub = g.sub;
    const i64 lda = g.lda, ldb = g.ldb, ldo = g.ldo;
    // split-K: slice blockIdx.y reduces k in [k_begin, k_end) into its own partial plane (rows not scattered).
    // Triangular B: only the k-range [k_lo, k_hi) of this column tile can hold non-zeros; it is what the slices share.
    int k_lo = 0, k_hi = K;
    if (g.tri == 1) k_hi = min(K, n0 + BN_);
    else if (g.tri == 2) k_lo = min(K, (n0 / BK_) * BK_);
    if (g.tri) k_chunk = (((k_hi - k_lo + (int)gridDim.y - 1) / (int)gridDim.y + BK_ - 1) / BK_) * BK_;
    const int k_begin = k_lo + blockIdx.y * k_chunk;
    const int k_end = min(k_hi, k_begin + k_chunk);
    const bool split = gridDim.y > 1;
    T* __restrict__ out = g.out + (i64)blockIdx.y * split_stride;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* As = reinterpret_cast<T*>(smem_raw);                       // [STAGES][BM][ALD]
    T* Bs = As + STAGES * A_STAGE;                                // [STAGES][BK][BLD]
    T* Ss = Bs + STAGES * B_STAGE;                                // [STAGES][BK_]  (sub vector slices)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp % WROWS) * (16 * MI), wn = (warp / WROWS) * (BN_ / 2);
    const int gq = lane >> 2, tq = lane & 3;
#ifdef B2H_GEMM_NO_STAGGER
    const bool early = true;
#else
    const bool early = warp < NT / 64;
#endif

    // Copy assignment, everything that does not depend on the k-tile computed once (the per-tile issue is ~6
    // instructions per 16-byte copy; the generic index arithmetic it replaces took 300 per k-tile and warp, executed by
    // every warp right after the barrier, i.e. with the tensor pipe idle).
    // A tile: BM rows x CPR chunks (16 B = 2 k); CPR consecutive threads take one row, NT / CPR rows per pass.
    constexpr int A_RPP = NT / CPR;
    const int a_kc = (tid % CPR) * 2;
    const T* a_ptr[A_ITERS];
    unsigned a_valid = 0;
#pragma unroll
    for (int i = 0; i < A_ITERS; ++i) {
        const int gr = m0 + tid / CPR + A_RPP * i;
        const bool ok = gr < M;
        a_ptr[i] = A + (ok ? (i64)(g.in_rows ? g.in_rows[gr] : gr) * lda : (i64)0);
        a_valid |= ok ? (1u << i) : 0u;
    }
    const unsigned a_dst = (unsigned)__cvta_generic_to_shared(As) + (unsigned)(((tid / CPR) * ALD_ + a_kc) * sizeof(T));
    // B tile: BK_ rows x BN_/2 chunks; 64 threads per row (those beyond the tile width idle), NT / 64 rows per pass.
    static_assert(BN_ / 2 <= 64, "B copy: one row per 64 threads");
    constexpr int B_RPP = NT / 64, B_ITERS = BK_ / B_RPP;
    const int b_col = (tid & 63) * 2, b_row = tid >> 6;
    const bool b_ok = b_col < BN_ && n0 + b_col < N;
    const T* b_ptr = B + (b_ok ? n0 + b_col : 0);
    const int ldb_i = (int)ldb;
    const unsigned b_dst = (unsigned)__cvta_generic_to_shared(Bs) + (unsigned)((b_row * BLD + b_col) * sizeof(T));

    auto issue = [&](int kt, int stage) {
        const int k0 = k_begin + kt * BK_;
        {
            const bool okk = k0 + a_kc < k_end;
            const int kofs = okk ? k0 + a_kc : 0;
            const unsigned dst = a_dst + (unsigned)(stage * A_STAGE * sizeof(T));
#pragma unroll
            for (int i = 0; i < A_ITERS; ++i)
                cp_async16s(dst + (unsigned)(i * A_RPP * ALD_ * sizeof(T)), a_ptr[i] + kofs,
                            (okk && ((a_valid >> i) & 1u)) ? 16 : 0);
        }
        {
            const unsigned dst = b_dst + (unsigned)(stage * B_STAGE * sizeof(T));
#pragma unroll
            for (int i = 0; i < B_ITERS; ++i) {
                const int gk = k0 + b_row + i * B_RPP;             // rows past the end of K: zero fill, address clamped
                cp_async16p(dst + (unsigned)(i * B_RPP * BLD * sizeof(T)), b_ptr + (i64)min(gk, k_end - 1) * ldb_i,
                            (b_ok && gk < k_end) ? 16 : 0, b_col < BN_);
            }
        }
        if (sub && tid < BK_ / 2) {
            const int gk = k0 + tid * 2;
            cp_async16(Ss + stage * BK_ + tid * 2, gk < k_end ? (const void*)(sub + gk) : (const void*)sub, gk < k_end ? 16 : 0);
        }
    };

    T acc[MI][NJ][4];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.0;

    const int nk = max((k_end - k_begin + BK_ - 1) / BK_, 0);
#pragma unroll
    for (int st = 0; st < STAGES - 1; ++st) {
        if (st < nk) issue(st, st);
        cp_async_commit();
    }
    for (int kt = 0; kt < nk; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();                                          // tile kt landed; buffer (kt-1)%STAGES is free
        auto refill = [&]() {
            const int nx = kt + STAGES - 1;
            if (nx < nk) issue(nx, nx % STAGES);
            cp_async_commit();
        };
        const int stage = kt % STAGES;
        const T* as = As + stage * A_STAGE + (wm + gq) * ALD_ + 2 * tq;
        const T* bs = Bs + stage * B_STAGE + (2 * tq) * BLD + wn;
        const T* ss = Ss + stage * BK_ + 2 * tq;
        constexpr int NP = NJ / 2;                                // column pairs of n8 tiles; NJ odd: one single tile
        // SUB: the launch subtracts a vector from the rows of A (the model's q - mu).  The subtraction runs on the
        // same FP64 pipe as the MMAs (ncu: a DADD waits for the pipe twice as long as a DMMA), so launches without a
        // vector -- two of the three contractions of a tick -- take a loop body without it.
        auto ktile = [&](auto sub_tag) {
            constexpr bool SUB = decltype(sub_tag)::value;
            T fa[MI][4], fb[NJ][2];
            // The two warps of a scheduler (w and w + NT / 64) refill the freed stage at different times: one right
            // after the barrier while the other already multiplies, the other in the middle of the k-tile -- the
            // copy-issue instructions of either run beside the other's MMAs instead of leaving the tensor pipe idle.
            if (early) refill();
#pragma unroll
            for (int s8 = 0; s8 < BK_ / 8; ++s8) {
                const int k0 = s8 * 8;
                double2 sv = make_double2(0.0, 0.0);
                if constexpr (SUB) sv = *reinterpret_cast<const double2*>(ss + k0);
#pragma unroll
                for (int i = 0; i < MI; ++i)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const double2 t = *reinterpret_cast<const double2*>(as + (i * 16 + h * 8) * ALD_ + k0);
                        fa[i][h] = SUB ? t.x - sv.x : t.x;        // k-slot tq     <- k0 + 2 tq
                        fa[i][2 + h] = SUB ? t.y - sv.y : t.y;    // k-slot tq + 4 <- k0 + 2 tq + 1
                    }
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const T* br = bs + (k0 + q) * BLD;
#pragma unroll
                    for (int pp = 0; pp < NP; ++pp) {
                        const double2 t = *reinterpret_cast<const double2*>(br + 16 * pp + 2 * gq);
                        fb[2 * pp][q] = t.x;
                        fb[2 * pp + 1][q] = t.y;
                    }
                    if constexpr (NJ & 1) fb[NJ - 1][q] = br[16 * NP + gq];
                }
                if (s8 == BK_ / 16 && !early) refill();
#pragma unroll
                for (int i = 0; i < MI; ++i)
#pragma unroll
                    for (int j = 0; j < NJ; ++j) Dmma<8>::run(acc[i][j], fa[i], fb[j]);
            }
        };
        // device-counted launches: a warp whose 32 rows lie past the row count only copies (the last 128-row tile of a
        // few hundred restarting chains is mostly empty)
        if (LOOP && m0 + wm >= M) refill();
        else if (sub) ktile(std::true_type{});
        else ktile(std::false_type{});
    }
    cp_async_wait<0>();

#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int gr = m0 + wm + i * 16 + h * 8 + gq;
            if (gr >= M) continue;
            const i64 orow = (i64)((g.out_rows && !split) ? g.out_rows[gr] : gr) * ldo;
            // tiles 2 p / 2 p + 1 hold the even / odd columns of group p: a lane owns 4 consecutive columns of it
#pragma unroll
            for (int pp = 0; pp < NJ / 2; ++pp) {
                const int gn = n0 + wn + 16 * pp + 4 * tq;
                if (gn < N)
                    *reinterpret_cast<double2*>(out + orow + gn) = make_double2(acc[i][2 * pp][2 * h], acc[i][2 * pp + 1][2 * h]);
                if (gn + 2 < N)
                    *reinterpret_cast<double2*>(out + orow + gn + 2) =
                        make_double2(acc[i][2 * pp][2 * h + 1], acc[i][2 * pp + 1][2 * h + 1]);
            }
            if constexpr (NJ & 1) {
                const int gn = n0 + wn + 16 * (NJ / 2) + tq * 2;
                if (gn < N)
                    *reinterpret_cast<double2*>(out + orow + gn) = make_double2(acc[i][NJ - 1][2 * h], acc[i][NJ - 1][2 * h + 1]);
            }
        }
    } while (LOOP && (tile += gridDim.x) < total_tiles);          // tiles of this CTA
}

template <int BN_, int MI, int BK_>
static void launch_async_v(cudaStream_t st, dim3 grid, int threads, const GemmGroup<double>& g0, const GemmGroup<double>& g1,
                           const GemmGroup<double>& g2, int N, int K, int tiles_n, int tiles_m0, int tiles_m1, int k_chunk,
                           i64 split_stride) {
    constexpr int smem = (STAGES * (BM * (BK_ + kApad) + BK_ * (BN_ + kBpad)) + STAGES * BK_) * (int)sizeof(double);
    const int total = (int)grid.x;
    if ((g0.M > 0 && g0.m_dev) || (g1.M > 0 && g1.m_dev) || (g2.M > 0 && g2.m_dev)) {
        static int sms = 0;
        if (sms == 0) {
            int dev = 0;
            cudaGetDevice(&dev);
            if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        }
        grid.x = (unsigned)std::max(1, std::min(total, (2 * sms + (int)grid.y - 1) / (int)grid.y));
        cudaFuncSetAttribute(dense_apply_dmma_async_kernel<BN_, MI, BK_, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        dense_apply_dmma_async_kernel<BN_, MI, BK_, true><<<grid, threads, smem, st>>>(g0, g1, g2, N, K, tiles_n, tiles_m0,
                                                                                       tiles_m1, k_chunk, split_stride, total);
        return;
    }
    cudaFuncSetAttribute(dense_apply_dmma_async_kernel<BN_, MI, BK_, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    dense_apply_dmma_async_kernel<BN_, MI, BK_, false><<<grid, threads, smem, st>>>(g0, g1, g2, N, K, tiles_n, tiles_m0,
                                                                                    tiles_m1, k_chunk, split_stride, total);
}

template <int BN_>
static void launch_async(cudaStream_t st, const GemmGroup<double>& g0, const GemmGroup<double>& g1,
                         const GemmGroup<double>& g2, int N, int K, int nsplit, int k_chunk, i64 split_stride) {
    int tiles_m0 = (g0.M + BM - 1) / BM, tiles_m1 = (g1.M + BM - 1) / BM, tiles_m2 = (g2.M + BM - 1) / BM;
    int tiles_n = (N + BN_ - 1) / BN_;
    dim3 grid((tiles_m0 + tiles_m1 + tiles_m2) * tiles_n, nsplit);
    static int warps = -1, bk = -1;
    if (warps < 0) { const char* e = getenv("B2H_GEMM_WARPS"); warps = e ? atoi(e) : B2H_GEMM_WARPS_DEFAULT; }
    if (bk < 0) { const char* e = getenv("B2H_GEMM_BK"); bk = e ? atoi(e) : B2H_GEMM_BK_DEFAULT; }
    if (warps == 16)
        launch_async_v<BN_, 1, 16>(st, grid, 512, g0, g1, g2, N, K, tiles_n, tiles_m0, tiles_m1, k_chunk, split_stride);
    else if (bk == 32)
        launch_async_v<BN_, 2, 32>(st, grid, 256, g0, g1, g2, N, K, tiles_n, tiles_m0, tiles_m1, k_chunk, split_stride);
    else
        launch_async_v<BN_, 2, 16>(st, grid, 256, g0, g1, g2, N, K, tiles_n, tiles_m0, tiles_m1, k_chunk, split_stride);
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }
static bool group_async_ok(const GemmGroup<double>& g) {
    if (g.M <= 0) return true;
    return aligned16(g.A) && aligned16(g.B) && aligned16(g.out) && (g.lda % 2 == 0) && (g.ldb % 2 == 0) &&
           (g.ldo % 2 == 0) && (!g.sub || aligned16(g.sub));
}

// pick the tile width whose tile count wastes the least of the last wave of 148 SMs
static int pick_bn(int M0, int rider_tile_rows, int N) {
    const int cand[3] = {128, 112, 96};
    int best = 128;
    double best_cost = 1e300;
    for (int c = 0; c < 3; ++c) {
        const int bn = cand[c];
        const long tiles = (long)((M0 + BM - 1) / BM + rider_tile_rows) * ((N + bn - 1) / bn);
        const long waves = (tiles + 147) / 148;
        const double cost = (double)waves * bn;        // time ~ waves x tile work
        if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
    }
    return best;
}

template <typename T>
static void launch_tile_kernel(dim3 grid, cudaStream_t st, const GemmGroup<T>& g0, const GemmGroup<T>& g1,
                               const GemmGroup<T>& g2, int N, int K, int tiles_n, int tiles_m0, int tiles_m1, int k_chunk,
                               i64 split_stride, int extra_rows_hint);

template <>
void launch_tile_kernel<double>(dim3 grid, cudaStream_t st, const GemmGroup<double>& g0, const GemmGroup<double>& g1,
                                const GemmGroup<double>& g2, int N, int K, int tiles_n, int tiles_m0, int tiles_m1,
                                int k_chunk, i64 split_stride, int extra_rows_hint) {
    static int use_async = -1;
    if (use_async < 0) {
        const char* e = getenv("B2H_GEMM_ASYNC");
        use_async = e ? atoi(e) : 1;
    }
    if (use_async && N % 2 == 0 && K % 2 == 0 && k_chunk % 2 == 0 && split_stride % 2 == 0 && group_async_ok(g0) &&
        group_async_ok(g1) && group_async_ok(g2)) {
        static int force_bn = -1;
        if (force_bn < 0) { const char* e = getenv("B2H_GEMM_BN"); force_bn = e ? atoi(e) : 0; }
        // the rider groups' row counts live on the device: the caller passes the expected number of rider TILE ROWS
        const int bn = force_bn ? force_bn : pick_bn(g0.M, extra_rows_hint, N);
        if (bn == 112) launch_async<112>(st, g0, g1, g2, N, K, grid.y, k_chunk, split_stride);
        else if (bn == 96) launch_async<96>(st, g0, g1, g2, N, K, grid.y, k_chunk, split_stride);
        else launch_async<128>(st, g0, g1, g2, N, K, grid.y, k_chunk, split_stride);
        return;
    }
    constexpr int smem = 2 * 2 * BK * DLD * (int)sizeof(double);
    static int ki = 0;
    if (ki == 0) {
        const char* e = getenv("B2H_DMMA_K");
        ki = e ? atoi(e) : 8;
    }
#define B2H_DMMA_LAUNCH(KI)                                                                                    \
    cudaFuncSetAttribute(dense_apply_dmma_kernel<KI>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);        \
    dense_apply_dmma_kernel<KI><<<grid, GT, smem, st>>>(g0, g1, g2, N, K, tiles_n, tiles_m0, tiles_m1, k_chunk, split_stride);
    if (ki == 4) { B2H_DMMA_LAUNCH(4) }
    else if (ki == 16) { B2H_DMMA_LAUNCH(16) }
    else { B2H_DMMA_LAUNCH(8) }
#undef B2H_DMMA_LAUNCH
}

template <>
void launch_tile_kernel<float>(dim3 grid, cudaStream_t st, const GemmGroup<float>& g0, const GemmGroup<float>& g1,
                               const GemmGroup<float>& g2, int N, int K, int tiles_n, int tiles_m0, int tiles_m1,
                               int k_chunk, i64 split_stride, int extra_rows_hint) {
    (void)extra_rows_hint;
    constexpr int smem = 2 * BK * (BM + BN) * (int)sizeof(float);
    cudaFuncSetAttribute(dense_apply_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    dense_apply_kernel<float><<<grid, GT, smem, st>>>(g0, g1, g2, N, K, tiles_n, tiles_m0, tiles_m1, k_chunk, split_stride);
}

// Up to three problems in one launch (riders may be empty: M == 0).  rider_tile_rows: expected number of 128-row
// tiles the riders will really occupy (their row counts live on the device), used to pick the tile width.
template <typename T>
void launch_gemm_grouped(cudaStream_t st, const GemmGroup<T>& g0, const GemmGroup<T>& g1, const GemmGroup<T>& g2, int N,
                         int K, int nsplit, i64 split_stride, int rider_tile_rows) {
    int tiles_m0 = (g0.M + BM - 1) / BM, tiles_m1 = (g1.M + BM - 1) / BM, tiles_m2 = (g2.M + BM - 1) / BM;
    int tiles_n = (N + BN - 1) / BN;
    if (tiles_m0 + tiles_m1 + tiles_m2 <= 0 || N <= 0) return;
    if (nsplit < 1) nsplit = 1;
    int k_chunk = (K + nsplit - 1) / nsplit;
    k_chunk = ((k_chunk + BK - 1) / BK) * BK;
    dim3 grid((tiles_m0 + tiles_m1 + tiles_m2) * tiles_n, nsplit);
    launch_tile_kernel<T>(grid, st, g0, g1, g2, N, K, tiles_n, tiles_m0, tiles_m1, k_chunk, split_stride, rider_tile_rows);
}

// General strided form with split-K: slice s of nsplit writes out + s*split_stride (a partial plane).
template <typename T>
void launch_gemm(cudaStream_t st, const T* A, i64 lda, const T* B, i64 ldb, T* out, i64 ldo, int M, int N, int K,
                 const int* m_dev, const T* sub, int nsplit, i64 split_stride) {
    if (M <= 0 || N <= 0) return;
    GemmGroup<T> g0{A, lda, B, ldb, out, ldo, M, m_dev, sub, nullptr, nullptr};
    GemmGroup<T> g1{nullptr, 0, nullptr, 0, nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr};
    launch_gemm_grouped<T>(st, g0, g1, g1, N, K, nsplit, split_stride, 0);
}

// out = (A - sub) . B ; sub (optional, [K]) is subtracted from every row of A on load (q - mu).
template <typename T>
void launch_dense_apply(cudaStream_t st, const T* A, const T* B, T* out, int M, int N, int K, const int* m_dev,
                        const T* sub) {
    launch_gemm<T>(st, A, (i64)K, B, (i64)N, out, (i64)N, M, N, K, m_dev, sub, 1, 0);
}

#define B2H_INST(T)                                                                                                  \
    template void launch_gemm_grouped<T>(cudaStream_t, const GemmGroup<T>&, const GemmGroup<T>&, const GemmGroup<T>&,  \
                                         int, int, int, i64, int);                                                    \
    template void launch_gemm<T>(cudaStream_t, const T*, i64, const T*, i64, T*, i64, int, int, int, const int*,     \
                                 const T*, int, i64);                                                                \
    template void launch_dense_apply<T>(cudaStream_t, const T*, const T*, T*, int, int, int, const int*, const T*);
B2H_INST(float)
B2H_INST(double)

template <typename T>
static GemmGroup<T> to_group(const b2h_gemm_group* g) {
    if (!g) return GemmGroup<T>{nullptr, 0, nullptr, 0, nullptr, 0, 0, nullptr, nullptr, nullptr, nullptr};
    return GemmGroup<T>{(const T*)g->A, g->lda, (const T*)g->B, g->ldb, (T*)g->out, g->ldo, (int)g->M,
                        (const int*)g->m_dev, (const T*)g->sub, nullptr, nullptr, g->tri};
}

template <typename T>
static void gemm_entry(cudaStream_t st, const b2h_gemm_group* g, int n, int N, int K, int nsplit, i64 split_stride) {
    launch_gemm_grouped<T>(st, to_group<T>(g), to_group<T>(n > 1 ? g + 1 : nullptr), to_group<T>(n > 2 ? g + 2 : nullptr),
                           N, K, nsplit, split_stride, 0);
}

}  // namespace b2h

extern "C" int b2h_gemm(b2h_ctx* ctx, int dtype, const b2h_gemm_group* groups, int32_t n_groups, int64_t N, int64_t K,
                        int32_t nsplit, int64_t split_stride) {
    using namespace b2h;
    if (!ctx) { set_error("null context"); return B2H_ERR_ARG; }
    if (dtype != B2H_F32 && dtype != B2H_F64) { set_error("bad dtype"); return B2H_ERR_ARG; }
    if (!groups || n_groups < 1 || n_groups > 3) { set_error("b2h_gemm: n_groups must be in [1, 3]"); return B2H_ERR_ARG; }
    if (N < 1 || K < 1 || nsplit < 1 || N > INT_MAX || K > INT_MAX) {
        set_error("b2h_gemm: N, K and nsplit must be in [1, INT_MAX]");
        return B2H_ERR_ARG;
    }
    for (int i = 0; i < n_groups; ++i) {
        const b2h_gemm_group& g = groups[i];
        if (g.M < 0 || g.M > INT_MAX || g.lda < K || g.ldb < N || g.ldo < N) {
            set_error("b2h_gemm: need 0 <= M <= INT_MAX, lda >= K, ldb >= N and ldo >= N");
            return B2H_ERR_ARG;
        }
        if (g.M > 0 && (!g.A || !g.B || !g.out)) { set_error("b2h_gemm: null matrix pointer"); return B2H_ERR_ARG; }
        if (g.tri < 0 || g.tri > 2) { set_error("b2h_gemm: tri must be 0, 1 or 2"); return B2H_ERR_ARG; }
    }
    if (dtype == B2H_F64) gemm_entry<double>(ctx->stream, groups, n_groups, (int)N, (int)K, nsplit, split_stride);
    else gemm_entry<float>(ctx->stream, groups, n_groups, (int)N, (int)K, nsplit, split_stride);
    B2H_LAUNCH_CHECK();
    return 0;
}
