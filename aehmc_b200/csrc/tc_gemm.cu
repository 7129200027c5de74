// tcgen05 / TMA tensor-core contraction for the batched logistic-regression gradient (config 3 / 5).
//
//   D[M x N] (fp32) = sum_{p < pieces} A_p[M x K] . B[N x K]^T        A_p, B: bf16, K-major (row-major, K contiguous)
//
// The gradient of all chains is two such products (SURVEY.md section 8d):
//   S[C x n] = sum_p Beta_p[C x D] . X[n x D]^T          (Beta split into 3 bf16 pieces: exact to 24 bits)
//   G[C x D] = sum_p R_p[C x n]    . Xt[D x n]^T         (R = sigmoid(S) - y split into 3 bf16 pieces)
// X is bf16-representable by construction, so every product is exact and accumulation is fp32 in TMEM: the result
// has fp32-class accuracy, which is what the float32 parity bar (1e-4) needs; the FMA path stays the exactness
// reference.
//
// Kernel anatomy (persistent: one CTA per SM loops over 128 x 128 output tiles, optional split-K planes; the
// accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the loads and MMAs of tile i+1):
//   warp 0 : TMA producer  -- cp.async.bulk.tensor 2D loads of 128 x 64 bf16 boxes (SWIZZLE_128B) into a 6-stage ring
//   warp 1 : MMA issuer    -- one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M128 N128 K16) from smem
//                             descriptors, tcgen05.commit releases the smem stage / signals the epilogue
//   warp 2 : TMEM allocator (128 columns)
//   warps 4-19: epilogue   -- tcgen05.ld 32x32b.x32 (TMEM lane quadrant = warp % 4, four warps per quadrant take
//                             32 of the 128 columns each: the epilogue is latency-bound, so it needs the warps); either fp32 -> global, or (logistic mode) the residual
//                             r = sigmoid(s) - y split into three bf16 pieces plus the potential's partial sums,
//                             so S is never written to memory
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "launch.h"

namespace b2h {

int logistic_fused_planes(int M, int N);

namespace tc {

constexpr int BM = 128, BN = 128, BK = 64;          // BK bf16 = one 128-byte swizzle row
constexpr int STAGES = 6;
constexpr int UMMA_K = 16;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int THREADS = 640;                        // warps 0-3: TMA / MMA / TMEM alloc / idle; warps 4-19: epilogue
constexpr int EPI_WARPS = 16, EPI_PARTS = EPI_WARPS / 4;   // 4 warps per TMEM lane quadrant, 32 columns each
constexpr int TMEM_COLS = 256;                      // two 128-column fp32 accumulators
constexpr size_t smem_bytes(int stages) { return (size_t)stages * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/; }

struct Epilogue {                 // mode 0: fp32 store.  mode 1: logistic residual pieces
    int mode;
    const float* y;               // [N] responses of this chunk
    __nv_bfloat16* r;             // residual pieces, TILE-BLOCKED: [3][column tile][row tile][128][128] bf16, so that
                                  // every 128 x 128 tile is one contiguous 32 KB block (DRAM-friendly writes)
    long long piece_stride;       // elements between pieces
    int tiles_m;                  // row tiles per column tile
    double* upart;                // [2 * gridDim.x][M] partial sums of softplus(s) - y s
};

__device__ __forceinline__ uint32_t pack_bf16(__nv_bfloat16 lo, __nv_bfloat16 hi) {
    return (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    }
}
// spin with a short sleep: for waits that are expected to be long (a spinning warp steals issue slots from the
// epilogue warps that share its scheduler)
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done = 0;
    while (true) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) break;
        __nanosleep(40);
    }
}
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// packed f32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2, one issue slot for two lanes of work)
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b),
                       rc = *reinterpret_cast<unsigned long long*>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long*>(&a), rb = *reinterpret_cast<unsigned long long*>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2*>(&rd);
}
// rr + (-float(h)) in one f32 = f16 + f32 instruction (sm_100, FHADD) that reads h, negated, from its half of a packed
// word: no unpacking to f32 first.  Exact when h = fp16(rr), and +0 when rr is fp16-exact (not -(h - rr), which is -0).
__device__ __forceinline__ float sub_f16(float rr, __half h) {
    float d;
    asm("{\n.reg .b16 n;\nneg.f16 n, %1;\nadd.rn.f32.f16 %0, n, %2;\n}" : "=f"(d) : "h"(__half_as_ushort(h)), "f"(rr));
    return d;
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred P;\n"
        "elect.sync _|P, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, P;\n"
        "}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}

// K-major, SWIZZLE_128B shared-memory operand descriptor (sm_100 "version 1"): rows of 128 bytes, 8-row groups
// 1024 bytes apart (SBO), leading offset unused for swizzled K-major layouts.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);          // start address
    d |= (uint64_t)1 << 16;                              // leading byte offset (ignored)
    d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset
    d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                              // SWIZZLE_128B
    return d;
}

// instruction descriptor: D = F32, A = B = BF16, both K-major, N = 128, M = 128
constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// Epilogue of one 128 x 128 accumulator for one warp: TMEM lane quadrant q, 32-column part `part`.
__device__ __forceinline__ float epilogue_tile(uint32_t tmem_base, int buf, int q, int part, int lane, int m0, int n0,
                                              int z, int M, int N, float* out, int ldo, long long split_stride,
                                              const Epilogue& ep, uint64_t* tmem_empty_bar) {
    const int row = m0 + q * 32 + lane;
    const int c0 = part * 32;
    uint32_t r[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + c0);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    // the accumulator is in registers: hand the TMEM buffer back to the MMA warp before doing the math
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(tmem_empty_bar)) : "memory");
    if (row >= M) return 0.f;
    if (ep.mode == 0) {
        float* orow = out + (long long)z * split_stride + (long long)row * ldo + n0;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const int col = n0 + c0 + j;
            if (col + 3 < N) {
                *reinterpret_cast<float4*>(orow + c0 + j) =
                    make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                __uint_as_float(r[j + 3]));
            } else {
                for (int e = 0; e < 4; ++e)
                    if (col + e < N) orow[c0 + j + e] = __uint_as_float(r[j + e]);
            }
        }
        return 0.f;
    }
    // logistic residual: r = sigmoid(s) - y as three bf16 pieces (exact split), potential partial sums
    float uacc = 0.f;
    uint32_t p0[16], p1[16], p2[16];
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        const int col = n0 + c0 + j;
        // y is warp-uniform per column: one 128-bit load serves four columns
        float4 y4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (col + 3 < N) y4 = __ldg(reinterpret_cast<const float4*>(ep.y + col));
        else {
            if (col < N) y4.x = __ldg(ep.y + col);
            if (col + 1 < N) y4.y = __ldg(ep.y + col + 1);
            if (col + 2 < N) y4.z = __ldg(ep.y + col + 2);
        }
        const float yv[4] = {y4.x, y4.y, y4.z, y4.w};
        float rr[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            // hardware exp2/log2/rcp approximations (abs error ~1e-7 here)
            const float sv = __uint_as_float(r[j + e]);
            const float ex = __expf(-fabsf(sv));
            const float inv = __fdividef(1.f, 1.f + ex);
            const bool ok = col + e < N;
            uacc += ok ? fmaxf(sv, 0.f) + __logf(1.f + ex) - yv[e] * sv : 0.f;
            rr[e] = ok ? (sv >= 0.f ? inv : ex * inv) - yv[e] : 0.f;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            // exact three-way split, two columns per packed conversion
            const __nv_bfloat162 a = __floats2bfloat162_rn(rr[2 * h], rr[2 * h + 1]);
            const float2 af = __bfloat1622float2(a);
            const float r1x = rr[2 * h] - af.x, r1y = rr[2 * h + 1] - af.y;
            const __nv_bfloat162 b = __floats2bfloat162_rn(r1x, r1y);
            const float2 bf = __bfloat1622float2(b);
            const __nv_bfloat162 c = __floats2bfloat162_rn(r1x - bf.x, r1y - bf.y);
            p0[(j >> 1) + h] = *reinterpret_cast<const uint32_t*>(&a);
            p1[(j >> 1) + h] = *reinterpret_cast<const uint32_t*>(&b);
            p2[(j >> 1) + h] = *reinterpret_cast<const uint32_t*>(&c);
        }
    }
    __nv_bfloat16* dst = ep.r + (((long long)(n0 / BN) * ep.tiles_m + m0 / BM) * BM + (row - m0)) * BN + c0;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        *reinterpret_cast<uint4*>(dst + 8 * v) = make_uint4(p0[4 * v], p0[4 * v + 1], p0[4 * v + 2], p0[4 * v + 3]);
        *reinterpret_cast<uint4*>(dst + ep.piece_stride + 8 * v) =
            make_uint4(p1[4 * v], p1[4 * v + 1], p1[4 * v + 2], p1[4 * v + 3]);
        *reinterpret_cast<uint4*>(dst + 2 * ep.piece_stride + 8 * v) =
            make_uint4(p2[4 * v], p2[4 * v + 1], p2[4 * v + 2], p2[4 * v + 3]);
    }
    return uacc;
}

__global__ void __launch_bounds__(THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, float* out,
               int M, int N, int K, int pieces, int piece_rows, int ldo, int k_blocks_per_split, long long split_stride,
               int stages, int tiles_m, int tiles_n, int nsplit, int a_blocked, Epilogue ep) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* tiles = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = (uint64_t*)(tiles + (size_t)stages * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;              // [2]
    uint64_t* tmem_empty = tmem_full + 2;                  // [2]
    uint32_t* tmem_slot = (uint32_t*)(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kb_total = (K + BK - 1) / BK;
    const int total_tiles = tiles_m * tiles_n * nsplit;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    // tile -> (split plane z, m tile, n tile), n fastest
    auto decode = [&](int tile, int& z, int& m0, int& n0, int& kb_begin, int& n_kb) {
        z = tile / (tiles_m * tiles_n);
        const int rem = tile - z * tiles_m * tiles_n;
        m0 = (rem / tiles_n) * BM;
        n0 = (rem % tiles_n) * BN;
        kb_begin = z * k_blocks_per_split;
        n_kb = max(min(kb_total, kb_begin + k_blocks_per_split) - kb_begin, 0);
    };

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int g = 0;                                     // ring position, continues across tiles
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                int z, m0, n0, kb_begin, n_kb;
                decode(tile, z, m0, n0, kb_begin, n_kb);
                const int iters = n_kb * pieces;
                for (int it = 0; it < iters; ++it, ++g) {
                    const int s = g % stages, round = g / stages;
                    mbar_wait(&empty_bar[s], (round & 1) ^ 1);
                    const int p = it / n_kb, kb = kb_begin + it % n_kb;
                    uint8_t* a_dst = tiles + (size_t)s * STAGE_BYTES;
                    uint8_t* b_dst = a_dst + A_BYTES;
                    mbar_expect_tx(&full_bar[s], STAGE_BYTES);
                    if (a_blocked)   // A is tile-blocked [piece][k tile of 128][row tile][128][128]: box = half a tile row
                        tma_load_2d(a_dst, &map_a, &full_bar[s], (kb & 1) * BK,
                                    p * piece_rows + ((kb >> 1) * tiles_m) * BM + m0);
                    else
                        tma_load_2d(a_dst, &map_a, &full_bar[s], kb * BK, p * piece_rows + m0);
                    tma_load_2d(b_dst, &map_b, &full_bar[s], kb * BK, n0);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            int g = 0, local = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++local) {
                int z, m0, n0, kb_begin, n_kb;
                decode(tile, z, m0, n0, kb_begin, n_kb);
                const int iters = n_kb * pieces;
                const int buf = local & 1;
                mbar_wait(&tmem_empty[buf], ((local >> 1) & 1) ^ 1);     // epilogue drained this accumulator
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t tmem_d = tmem_base + (uint32_t)(buf * BN);
                for (int it = 0; it < iters; ++it, ++g) {
                    const int s = g % stages, round = g / stages;
                    mbar_wait(&full_bar[s], round & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_addr = smem_u32(tiles + (size_t)s * STAGE_BYTES);
                    const uint32_t b_addr = a_addr + A_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t ad = make_desc(a_addr + k * UMMA_K * 2);
                        const uint64_t bd = make_desc(b_addr + k * UMMA_K * 2);
                        umma_bf16(tmem_d, ad, bd, IDESC, (it > 0 || k > 0) ? 1u : 0u);
                    }
                    tcgen05_commit(&empty_bar[s]);         // frees the smem stage when these MMAs retire
                }
                tcgen05_commit(&tmem_full[buf]);           // accumulator complete
            }
        }
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers -> global =====
        const int q = warp & 3;                            // TMEM lane quadrant this warp may access
        const int half = (warp - 4) >> 2;                  // which 32 of the 128 accumulator columns
        int local = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++local) {
            int z, m0, n0, kb_begin, n_kb;
            decode(tile, z, m0, n0, kb_begin, n_kb);
            const int buf = local & 1;
            mbar_wait(&tmem_full[buf], (local >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const float u = epilogue_tile(tmem_base, buf, q, half, lane, m0, n0, z, M, N, out, ldo, split_stride, ep,
                                          &tmem_empty[buf]);
            const int row = m0 + q * 32 + lane;
            if (ep.mode == 1 && row < M) ep.upart[((long long)(n0 / BN) * EPI_PARTS + half) * M + row] = (double)u;
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// A-resident variant for short reductions (the S product: K = dim <= 128, so pieces * K/64 <= 6 blocks).
// All (piece, k-block) tiles of A for the CTA's current 128 rows stay in shared memory; the CTA walks a contiguous
// range of column tiles and streams each B tile (full K) exactly once through a 3-slot ring.  Operand traffic per
// output tile drops from pieces * 2 * K/64 * 16 KB to K/64 * 16 KB.
// ---------------------------------------------------------------------------------------------------------
constexpr int RES_A_BLOCKS = 6, RES_B_SLOTS = 3, RES_KB = 2;
constexpr size_t RES_SMEM = (size_t)RES_A_BLOCKS * A_BYTES + (size_t)RES_B_SLOTS * RES_KB * B_BYTES + 1024 + 256;

__global__ void __launch_bounds__(THREADS, 1)
tc_gemm_resident_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, float* out,
                        int M, int N, int K, int pieces, int piece_rows, int ldo, int tiles_m, int tiles_n,
                        int tiles_per_cta, Epilogue ep) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* a_res = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* b_ring = a_res + (size_t)RES_A_BLOCKS * A_BYTES;
    uint64_t* bars = (uint64_t*)(b_ring + (size_t)RES_B_SLOTS * RES_KB * B_BYTES);
    uint64_t* b_full = bars;                   // [3]
    uint64_t* b_empty = bars + 3;              // [3]
    uint64_t* a_full = bars + 6;               // [1]
    uint64_t* a_free = bars + 7;               // [1]
    uint64_t* tmem_full = bars + 8;            // [2]
    uint64_t* tmem_empty = bars + 10;          // [2]
    uint32_t* tmem_slot = (uint32_t*)(bars + 12);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kb_total = (K + BK - 1) / BK;                    // <= RES_KB
    const int total_tiles = tiles_m * tiles_n;
    const int t_begin = blockIdx.x * tiles_per_cta;
    const int t_end = min(total_tiles, t_begin + tiles_per_cta);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < 3; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
        mbar_init(a_full, 1); mbar_init(a_free, 1);
        for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int a_loads = 0, cur_m = -1;
            for (int tile = t_begin, local = 0; tile < t_end; ++tile, ++local) {
                const int m_tile = tile / tiles_n, n0 = (tile % tiles_n) * BN;
                if (m_tile != cur_m) {
                    // the previous rows' MMAs must have retired before A is overwritten
                    mbar_wait(a_free, (a_loads & 1) ^ 1);
                    mbar_expect_tx(a_full, (uint32_t)(pieces * kb_total * A_BYTES));
                    for (int p = 0; p < pieces; ++p)
                        for (int kb = 0; kb < kb_total; ++kb)
                            tma_load_2d(a_res + (size_t)(p * kb_total + kb) * A_BYTES, &map_a, a_full, kb * BK,
                                        p * piece_rows + m_tile * BM);
                    ++a_loads;
                    cur_m = m_tile;
                }
                const int slot = local % RES_B_SLOTS, round = local / RES_B_SLOTS;
                mbar_wait(&b_empty[slot], (round & 1) ^ 1);
                mbar_expect_tx(&b_full[slot], (uint32_t)(kb_total * B_BYTES));
                for (int kb = 0; kb < kb_total; ++kb)
                    tma_load_2d(b_ring + (size_t)(slot * RES_KB + kb) * B_BYTES, &map_b, &b_full[slot], kb * BK, n0);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int a_loads = 0, cur_m = -1;
            for (int tile = t_begin, local = 0; tile < t_end; ++tile, ++local) {
                const int m_tile = tile / tiles_n;
                if (m_tile != cur_m) {
                    mbar_wait(a_full, a_loads & 1);
                    ++a_loads;
                    cur_m = m_tile;
                }
                const int buf = local & 1;
                mbar_wait(&tmem_empty[buf], ((local >> 1) & 1) ^ 1);
                const int slot = local % RES_B_SLOTS, round = local / RES_B_SLOTS;
                mbar_wait(&b_full[slot], round & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t tmem_d = tmem_base + (uint32_t)(buf * BN);
                bool first = true;
                for (int p = 0; p < pieces; ++p)
                    for (int kb = 0; kb < kb_total; ++kb) {
                        const uint32_t a_addr = smem_u32(a_res + (size_t)(p * kb_total + kb) * A_BYTES);
                        const uint32_t b_addr = smem_u32(b_ring + (size_t)(slot * RES_KB + kb) * B_BYTES);
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k) {
                            umma_bf16(tmem_d, make_desc(a_addr + k * UMMA_K * 2), make_desc(b_addr + k * UMMA_K * 2), IDESC,
                                      first ? 0u : 1u);
                            first = false;
                        }
                    }
                tcgen05_commit(&b_empty[slot]);
                tcgen05_commit(&tmem_full[buf]);
                const bool last_of_rows = (tile + 1 >= t_end) || ((tile + 1) / tiles_n != m_tile);
                if (last_of_rows) tcgen05_commit(a_free);
            }
        }
    } else if (warp >= 4) {
        const int q = warp & 3, half = (warp - 4) >> 2;
        float urun = 0.f;                      // potential partial sum of this thread's row over the CTA's tiles
        for (int tile = t_begin, local = 0; tile < t_end; ++tile, ++local) {
            const int m0 = (tile / tiles_n) * BM, n0 = (tile % tiles_n) * BN;
            const int buf = local & 1;
            mbar_wait(&tmem_full[buf], (local >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            urun += epilogue_tile(tmem_base, buf, q, half, lane, m0, n0, 0, M, N, out, ldo, 0, ep, &tmem_empty[buf]);
            const bool last_of_rows = (tile + 1 >= t_end) || ((tile + 1) / tiles_n != tile / tiles_n);
            if (last_of_rows) {
                const int row = m0 + q * 32 + lane;
                if (ep.mode == 1 && row < M) ep.upart[((long long)blockIdx.x * EPI_PARTS + half) * M + row] = (double)urun;
                urun = 0.f;
            }
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}


// ---------------------------------------------------------------------------------------------------------
// Fully fused logistic gradient (dim <= 128): S and the residual never leave tensor memory.
//
// A work item is (chain tile of 128 chains, data tile of 64 rows); every CTA takes a contiguous range of items
// (data tile fastest) and for each item runs
//   MMA1 (warp 1)   S[128 c x 64 n]  = sum_p Beta_p[128 c x D] . X[64 n x D]^T   Beta pieces resident in shared memory,
//                                                                                X tile streamed once by TMA (6-stage ring)
//   epilogue (16 warps)  r = sigmoid(s) - y split exactly into three bf16 pieces and stored straight back to TENSOR
//                        MEMORY (tcgen05.st) as the A operand of the second product; potential partial sums in registers
//   MMA2 (warp 3)   G[128 c x D]    += sum_p R_p[128 c x 64 n] . X[64 n x D]     A from TMEM (no shared-memory traffic
//                                                                                for the residual), B = THE SAME X tile
//                                                                                read through an MN-major descriptor
// G accumulates in TMEM over the whole data range of the CTA and is written once per (CTA, chain tile) as an fp32
// partial plane; a small kernel sums the planes in a fixed order (deterministic).  The two products have separate
// issuing warps, so the first product runs ahead (bounded by the two S buffers) instead of queueing behind the
// residual hand-off of the previous item.  Why A-from-TMEM: with both operands in shared memory the kernel was bound
// by shared-memory bandwidth (an M128 N64 K16 step reads 6 KB in 32 tensor cycles, plus the epilogue's own stores).
// TMEM columns: [0,64) [64,128) = S double buffer, [128,256) = G, [256,352) [352,448) = residual pieces double buffer
// (per piece 32 columns: two bf16 data rows per 32-bit cell, lane = chain).
// ---------------------------------------------------------------------------------------------------------
constexpr int FN = 64;                                   // data rows per item
constexpr int F_XSTAGES = 6;
constexpr int F_XBOX = FN * BK * 2;                      // 8 KB: 64 rows x 64 features
constexpr int F_XSTAGE = 2 * F_XBOX;                     // 16 KB: both feature halves
constexpr int F_TMEM_COLS = 512;
constexpr uint32_t F_COL_G = 128, F_COL_R = 256, F_RBUF_COLS = 96, F_RPIECE_COLS = 32;
constexpr size_t F_SMEM = (size_t)RES_A_BLOCKS * A_BYTES + (size_t)F_XSTAGES * F_XSTAGE + 1024 + 512;
// instruction descriptors: D = F32, A = B = BF16.  MMA1: both K-major, N = 64.  MMA2: B MN-major (bit 16), N = 128.
constexpr uint32_t IDESC_S = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
constexpr uint32_t IDESC_G = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)(BM >> 4) << 24);

// MN-major SWIZZLE_128B operand: 128-byte rows hold 64 consecutive MN elements of one K index, 8 K rows per
// 1024-byte atom; LBO = distance between 64-element MN atoms, SBO = distance between 8-row K groups.
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// A operand in tensor memory (lane = row, two 16-bit K elements per 32-bit column)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
                 "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}

struct FusedArgs {
    const float* y;          // [N]
    float* gpart;            // [planes][M x dim] fp32 partial gradients
    long long plane_stride;  // M * dim
    double* upart;           // [gridDim.x][4][M] potential partial sums
    int M, N, dim, piece_rows, tiles_m, tiles_n, per_cta;
};

template <int KB>
__global__ void __launch_bounds__(THREADS, 1)
tc_logistic_fused_kernel(const __grid_constant__ CUtensorMap map_beta, const __grid_constant__ CUtensorMap map_x,
                         FusedArgs fa) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* a_res = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* x_ring = a_res + (size_t)RES_A_BLOCKS * A_BYTES;
    uint64_t* bars = (uint64_t*)(x_ring + (size_t)F_XSTAGES * F_XSTAGE);
    uint64_t* x_full = bars;                          // [6]
    uint64_t* x_empty = bars + F_XSTAGES;             // [6]
    uint64_t* a_full = bars + 2 * F_XSTAGES;
    uint64_t* a_free = a_full + 1;
    uint64_t* s_full = a_full + 2;                    // [2]
    uint64_t* s_empty = a_full + 4;                   // [2]
    uint64_t* r_full = a_full + 6;                    // [2]
    uint64_t* r_empty = a_full + 8;                   // [2]
    uint64_t* g_full = a_full + 10;
    uint64_t* g_empty = a_full + 11;
    uint32_t* tmem_slot = (uint32_t*)(a_full + 12);

    // the warp index goes through a shuffle so that the compiler treats role branches as warp-uniform
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int tiles_n = fa.tiles_n;
    const int total = fa.tiles_m * tiles_n;
    const int t_begin = blockIdx.x * fa.per_cta;
    const int t_end = min(total, t_begin + fa.per_cta);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_beta) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < F_XSTAGES; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
        mbar_init(a_full, 1); mbar_init(a_free, 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&s_full[b], 1); mbar_init(&s_empty[b], EPI_WARPS);
            mbar_init(&r_full[b], EPI_WARPS); mbar_init(&r_empty[b], 1);
        }
        mbar_init(g_full, 1); mbar_init(g_empty, EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(F_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        // ===== TMA producer: Beta pieces once per chain tile, one X tile per item =====
        if (lane == 0) {
            int a_loads = 0, cur_m = -1;
            int m_tile = t_begin / tiles_n, n_tile = t_begin - m_tile * tiles_n;
            for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
                if (m_tile != cur_m) {
                    mbar_wait(a_free, (a_loads & 1) ^ 1);      // first products of the previous chain tile retired
                    mbar_expect_tx(a_full, (uint32_t)(3 * KB * A_BYTES));
                    for (int p = 0; p < 3; ++p)
                        for (int kb = 0; kb < KB; ++kb)
                            tma_load_2d(a_res + (size_t)(p * KB + kb) * A_BYTES, &map_beta, a_full, kb * BK,
                                        p * fa.piece_rows + m_tile * BM);
                    ++a_loads;
                    cur_m = m_tile;
                }
                const int s = L % F_XSTAGES, round = L / F_XSTAGES;
                mbar_wait_backoff(&x_empty[s], (round & 1) ^ 1);
                mbar_expect_tx(&x_full[s], (uint32_t)(KB * F_XBOX));
                for (int kb = 0; kb < KB; ++kb)
                    tma_load_2d(x_ring + (size_t)s * F_XSTAGE + (size_t)kb * F_XBOX, &map_x, &x_full[s], kb * BK, n_tile * FN);
                if (++n_tile == tiles_n) { n_tile = 0; ++m_tile; }
            }
        }
    } else if (warp == 1) {
        // ===== issuer of the first product.  The whole warp runs the loop (warp-uniform control flow keeps the operand
        // descriptors in uniform registers), one elected lane issues: with a single diverged lane every tcgen05.mma
        // cost ~15 dependent instructions of descriptor arithmetic and the issuer paced the kernel. =====
        const uint64_t a_desc0 = make_desc(smem_u32(a_res));
        const uint32_t x_ring_addr = smem_u32(x_ring);
        int a_loads = 0, cur_m = -1;
        int m_tile = t_begin / tiles_n, n_tile = t_begin - m_tile * tiles_n;
        for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
            if (m_tile != cur_m) {
                mbar_wait(a_full, a_loads & 1);
                ++a_loads;
                cur_m = m_tile;
            }
            const int buf = L & 1;
            const int stage = L % F_XSTAGES;
            mbar_wait(&s_empty[buf], ((L >> 1) & 1) ^ 1);
            mbar_wait(&x_full[stage], (L / F_XSTAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t tmem_s = tmem_base + (uint32_t)(buf * FN);
            const uint64_t xd = make_desc(x_ring_addr + (uint32_t)stage * F_XSTAGE);
            const bool last_of_seg = (t + 1 >= t_end) || (n_tile + 1 == tiles_n);
            if (elect_one()) {
#pragma unroll
                for (int p = 0; p < 3; ++p)
#pragma unroll
                    for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k)
                            umma_bf16(tmem_s, a_desc0 + (uint64_t)(((p * KB + kb) * A_BYTES + k * UMMA_K * 2) >> 4),
                                      xd + (uint64_t)((kb * F_XBOX + k * UMMA_K * 2) >> 4), IDESC_S,
                                      (p == 0 && kb == 0 && k == 0) ? 0u : 1u);
                tcgen05_commit(&s_full[buf]);
                if (last_of_seg) tcgen05_commit(a_free);
            }
            __syncwarp();
            if (++n_tile == tiles_n) { n_tile = 0; ++m_tile; }
        }
    } else if (warp == 3) {
        // ===== issuer of the second product: A = residual pieces in tensor memory, B = the item's X tile (MN-major) =====
        const uint32_t x_ring_addr = smem_u32(x_ring);
        const uint32_t tmem_g = tmem_base + F_COL_G;
        int segs_done = 0;
        int m_tile = t_begin / tiles_n, n_tile = t_begin - m_tile * tiles_n;
        bool first_of_seg = true;
        for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
            const bool last_of_seg = (t + 1 >= t_end) || (n_tile + 1 == tiles_n);
            const int rb = L & 1, stage = L % F_XSTAGES;
            mbar_wait(&r_full[rb], (L >> 1) & 1);
            mbar_wait(&x_full[stage], (L / F_XSTAGES) & 1);               // already complete; orders this warp after the TMA
            if (first_of_seg && segs_done > 0) mbar_wait(g_empty, (segs_done - 1) & 1);   // G drained
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t xd = make_desc_mn(x_ring_addr + (uint32_t)stage * F_XSTAGE, F_XBOX, 1024);
            const uint32_t tmem_r = tmem_base + F_COL_R + (uint32_t)rb * F_RBUF_COLS;
            if (elect_one()) {
#pragma unroll
                for (int p = 0; p < 3; ++p)
#pragma unroll
                    for (int k = 0; k < FN / UMMA_K; ++k)
                        umma_bf16_ts(tmem_g, tmem_r + (uint32_t)(p * F_RPIECE_COLS + k * (UMMA_K / 2)),
                                     xd + (uint64_t)((k * UMMA_K * 128) >> 4), IDESC_G,
                                     (first_of_seg && p == 0 && k == 0) ? 0u : 1u);
                tcgen05_commit(&x_empty[stage]);
                tcgen05_commit(&r_empty[rb]);
                if (last_of_seg) tcgen05_commit(g_full);
            }
            __syncwarp();
            first_of_seg = last_of_seg;
            if (last_of_seg) ++segs_done;
            if (++n_tile == tiles_n) { n_tile = 0; ++m_tile; }
        }
    } else if (warp >= 4) {
        // ===== epilogue warps: S -> residual pieces back into tensor memory; G -> partial plane at the end of a segment =====
        const int q = warp & 3, part = (warp - 4) >> 2;
        const int trow = q * 32 + lane;                        // row of the 128-chain tile = TMEM lane
        const int c0 = part * 16;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        float urun = 0.f;
        int segs_done = 0;
        int m_tile = t_begin / tiles_n, n_tile = t_begin - m_tile * tiles_n;
        for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
            const int n0 = n_tile * FN;
            const int buf = L & 1;
            const bool full = n0 + FN <= fa.N;
            // responses of this thread's 16 data rows (warp-uniform addresses), requested before S is waited for
            float yv[16];
            if (full) {
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                    const float4 y4 = __ldg(reinterpret_cast<const float4*>(fa.y + n0 + c0 + j));
                    yv[j] = y4.x; yv[j + 1] = y4.y; yv[j + 2] = y4.z; yv[j + 3] = y4.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) yv[j] = (n0 + c0 + j < fa.N) ? __ldg(fa.y + n0 + c0 + j) : 0.5f;
            }
            mbar_wait_backoff(&s_full[buf], (L >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t r[16];
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                  "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                : "r"(lane_addr + (uint32_t)(buf * FN + c0)));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&s_empty[buf])) : "memory");

            uint32_t p0[8], p1[8], p2[8];
            float uacc;
            {
                // MUFU is a quarter-rate pipe and this loop is its only user, so the special functions are batched:
                // one ex2 per element, one rcp per PAIR (1/a = b / (a b)) and one lg2 per 16 elements (sum of logs =
                // log of the product; every factor is in (1, 2], the product <= 65536); truncating split.
                float rr[16], den[16];
                float ua0 = 0.f, ua1 = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float sv = __uint_as_float(r[j]);
                    const float ex = ex2_approx(fabsf(sv) * -1.4426950408889634f);
                    den[j] = 1.f + ex;
                    rr[j] = sv >= 0.f ? 1.f : ex;                            // numerator of sigmoid(s)
                    if (j & 1) ua1 += fmaf(-yv[j], sv, fmaxf(sv, 0.f));
                    else ua0 += fmaf(-yv[j], sv, fmaxf(sv, 0.f));
                }
                float pp[8];
#pragma unroll
                for (int h = 0; h < 8; ++h) {
                    pp[h] = den[2 * h] * den[2 * h + 1];
                    const float rp = rcp_approx(pp[h]);
                    rr[2 * h] = fmaf(rr[2 * h], den[2 * h + 1] * rp, -yv[2 * h]);
                    rr[2 * h + 1] = fmaf(rr[2 * h + 1], den[2 * h] * rp, -yv[2 * h + 1]);
                }
                const float prod = ((pp[0] * pp[1]) * (pp[2] * pp[3])) * ((pp[4] * pp[5]) * (pp[6] * pp[7]));
                uacc = fmaf(lg2_approx(prod), 0.6931471805599453f, ua0 + ua1);
#pragma unroll
                for (int h = 0; h < 8; ++h) {
                    // exact three-way split by truncation (8 + 8 + 8 significant bits), two data rows per packed word
                    const uint32_t a0 = __float_as_uint(rr[2 * h]), b0 = __float_as_uint(rr[2 * h + 1]);
                    const float a1 = rr[2 * h] - __uint_as_float(a0 & 0xffff0000u);
                    const float b1 = rr[2 * h + 1] - __uint_as_float(b0 & 0xffff0000u);
                    const uint32_t a1u = __float_as_uint(a1), b1u = __float_as_uint(b1);
                    const float a2 = a1 - __uint_as_float(a1u & 0xffff0000u);
                    const float b2 = b1 - __uint_as_float(b1u & 0xffff0000u);
                    p0[h] = __byte_perm(a0, b0, 0x7632);
                    p1[h] = __byte_perm(a1u, b1u, 0x7632);
                    p2[h] = __byte_perm(__float_as_uint(a2), __float_as_uint(b2), 0x7632);
                }
            }
            // rows past the end of the data (s = 0 from the zero-filled X rows, y loaded as 1/2): the residual is
            // 0 by construction and each such row added log 2 to the potential
            if (!full) uacc -= 0.6931471805599453f * (float)min(16, max(0, n0 + c0 + 16 - fa.N));
            urun += uacc;
            // residual pieces -> tensor memory (the second product of item L - 2 must have consumed this buffer)
            {
                const int rb = L & 1;
                mbar_wait(&r_empty[rb], ((L >> 1) & 1) ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t raddr = lane_addr + F_COL_R + (uint32_t)rb * F_RBUF_COLS + (uint32_t)(part * 8);
                tmem_st8(raddr, p0);
                tmem_st8(raddr + F_RPIECE_COLS, p1);
                tmem_st8(raddr + 2 * F_RPIECE_COLS, p2);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&r_full[rb])) : "memory");
            }

            const bool last_of_seg = (t + 1 >= t_end) || (n_tile + 1 == tiles_n);
            if (last_of_seg) {
                // drain G: this warp's lane quadrant, columns [32 part, 32 part + 32)
                mbar_wait(g_full, segs_done & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                uint32_t gq[32];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(gq[0]), "=r"(gq[1]), "=r"(gq[2]), "=r"(gq[3]), "=r"(gq[4]), "=r"(gq[5]), "=r"(gq[6]), "=r"(gq[7]),
                      "=r"(gq[8]), "=r"(gq[9]), "=r"(gq[10]), "=r"(gq[11]), "=r"(gq[12]), "=r"(gq[13]), "=r"(gq[14]),
                      "=r"(gq[15]), "=r"(gq[16]), "=r"(gq[17]), "=r"(gq[18]), "=r"(gq[19]), "=r"(gq[20]), "=r"(gq[21]),
                      "=r"(gq[22]), "=r"(gq[23]), "=r"(gq[24]), "=r"(gq[25]), "=r"(gq[26]), "=r"(gq[27]), "=r"(gq[28]),
                      "=r"(gq[29]), "=r"(gq[30]), "=r"(gq[31])
                    : "r"(lane_addr + F_COL_G + (uint32_t)(part * 32)));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(g_empty)) : "memory");
                ++segs_done;
                const int row = m_tile * BM + trow;
                if (row < fa.M) {
                    // plane = position of this CTA among the CTAs that touch the chain tile
                    const int b_first = (int)(((long long)m_tile * tiles_n) / fa.per_cta);
                    float* orow = fa.gpart + (long long)(blockIdx.x - b_first) * fa.plane_stride + (long long)row * fa.dim;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const int col = part * 32 + j;
                        if (col + 3 < fa.dim) {
                            *reinterpret_cast<float4*>(orow + col) =
                                make_float4(__uint_as_float(gq[j]), __uint_as_float(gq[j + 1]), __uint_as_float(gq[j + 2]),
                                            __uint_as_float(gq[j + 3]));
                        } else {
                            for (int e = 0; e < 4; ++e)
                                if (col + e < fa.dim) orow[col + e] = __uint_as_float(gq[j + e]);
                        }
                    }
                    fa.upart[((long long)blockIdx.x * EPI_PARTS + part) * fa.M + row] = (double)urun;
                }
                urun = 0.f;
            }
            if (++n_tile == tiles_n) { n_tile = 0; ++m_tile; }
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(F_TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// fp16 x 2 variant of the fused gradient: beta and the residual are carried as TWO fp16 pieces (22 significant
// bits; the hardware does not mix an fp16 A with a bf16 B inside kind::f16, so X is read from an exact fp16 copy
// X * 2^shift).  Two thirds of the tensor work of the bf16 x 3 kernel, and small enough for BOTH products to take
// their A operand from tensor memory: the beta pieces of the CTA's chain tile are stored to TMEM once per segment by
// the epilogue warps, so shared memory carries nothing but the X ring.
// Scales (powers of two, exact): X holds X * 2^shift, the beta pieces hold beta * 2^(20 - shift), so S_acc = s * 2^20;
// the residual pieces hold r itself (the low piece may be an fp16 subnormal: absolute error <= 2^-25, what an fp32
// residual has anyway), so G_acc = g * 2^shift.
// TMEM columns: [0,128) S double buffer, [128,256) G, [256,384) residual double buffer (2 x 2 pieces x 32),
// [384,512) beta (2 pieces x 64).
// ---------------------------------------------------------------------------------------------------------
constexpr int H_XSTAGES = 8;
constexpr uint32_t H_COL_R = 256, H_RBUF_COLS = 64, H_RPIECE_COLS = 32, H_COL_B = 384, H_BPIECE_COLS = 64;
constexpr size_t H_SMEM = (size_t)H_XSTAGES * F_XSTAGE + 1024 + 512;
constexpr uint32_t IDESC_S16 = (1u << 4) | ((uint32_t)(FN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
constexpr uint32_t IDESC_G16 = (1u << 4) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

struct Fused16Args {
    const float* y;          // [N] responses
    const __half* beta;      // [2][M x dim] fp16 pieces of beta * 2^(acc_exp - shift)
    float* gpart;            // [planes][M x dim] fp32 partial gradients (scaled by 2^shift)
    long long plane_stride;  // M * dim
    double* upart;           // [gridDim.x][4][M] potential partial sums
    float s_scale;           // 2^-acc_exp: accumulator -> s
    int M, N, dim, tiles_m, tiles_n, per_cta;
};

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}

template <int KB>
__global__ void __launch_bounds__(THREADS, 1)
tc_logistic_fused16_kernel(const __grid_constant__ CUtensorMap map_x, Fused16Args fa) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* x_ring = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(x_ring + (size_t)H_XSTAGES * F_XSTAGE);
    uint64_t* x_full = bars;                          // [8]
    uint64_t* x_empty = bars + H_XSTAGES;             // [8]
    uint64_t* a_full = bars + 2 * H_XSTAGES;
    uint64_t* a_free = a_full + 1;
    uint64_t* s_full = a_full + 2;                    // [2]
    uint64_t* s_empty = a_full + 4;                   // [2]
    uint64_t* r_full = a_full + 6;                    // [2]
    uint64_t* r_empty = a_full + 8;                   // [2]
    uint64_t* g_full = a_full + 10;
    uint64_t* g_empty = a_full + 11;
    uint32_t* tmem_slot = (uint32_t*)(a_full + 12);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int tiles_n = fa.tiles_n;
    const int total = fa.tiles_m * tiles_n;
    const int t_begin = blockIdx.x * fa.per_cta;
    const int t_end = min(total, t_begin + fa.per_cta);

    if (warp == 0 && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < H_XSTAGES; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
        mbar_init(a_full, EPI_WARPS); mbar_init(a_free, 1);
        for (int b = 0; b < 2; ++b) {
            mbar_init(&s_full[b], 1); mbar_init(&s_empty[b], EPI_WARPS);
            mbar_init(&r_full[b], EPI_WARPS); mbar_init(&r_empty[b], 1);
        }
        mbar_init(g_full, 1); mbar_init(g_empty, EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(F_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

    if (warp == 0) {
        // ===== TMA producer: one X tile per item =====
        if (lane == 0) {
            int n_tile = t_begin % tiles_n;
            for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
                const int s = L % H_XSTAGES, round = L / H_XSTAGES;
                mbar_wait_backoff(&x_empty[s], (round & 1) ^ 1);
                mbar_expect_tx(&x_full[s], (uint32_t)(KB * F_XBOX));
                for (int kb = 0; kb < KB; ++kb)
                    tma_load_2d(x_ring + (size_t)s * F_XSTAGE + (size_t)kb * F_XBOX, &map_x, &x_full[s], kb * BK, n_tile * FN);
                if (++n_tile == tiles_n) n_tile = 0;
            }
        }
    } else if (warp == 1) {
        // ===== issuer of the first product: A = beta pieces in tensor memory, B = X tile (K-major) =====
        const uint32_t x_ring_addr = smem_u32(x_ring);
        const uint32_t tmem_b = tmem_base + H_COL_B;
        int seg = 0;
        int n_tile = t_begin % tiles_n;
        bool first_of_seg = true;
        for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
            if (first_of_seg) { mbar_wait(a_full, seg & 1); ++seg; }
            const int buf = L & 1;
            const int stage = L % H_XSTAGES;
            mbar_wait(&s_empty[buf], ((L >> 1) & 1) ^ 1);
            mbar_wait(&x_full[stage], (L / H_XSTAGES) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t tmem_s = tmem_base + (uint32_t)(buf * FN);
            const uint64_t xd = make_desc(x_ring_addr + (uint32_t)stage * F_XSTAGE);
            const bool last_of_seg = (t + 1 >= t_end) || (n_tile + 1 == tiles_n);
            if (elect_one()) {
#pragma unroll
                for (int p = 0; p < 2; ++p)
#pragma unroll
                    for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                        for (int k = 0; k < BK / UMMA_K; ++k)
                            umma_bf16_ts(tmem_s, tmem_b + (uint32_t)(p * H_BPIECE_COLS + kb * (BK / 2) + k * (UMMA_K / 2)),
                                         xd + (uint64_t)((kb * F_XBOX + k * UMMA_K * 2) >> 4), IDESC_S16,
                                         (p == 0 && kb == 0 && k == 0) ? 0u : 1u);
                tcgen05_commit(&s_full[buf]);
                if (last_of_seg) tcgen05_commit(a_free);
            }
            __syncwarp();
            first_of_seg = last_of_seg;
            if (++n_tile == tiles_n) n_tile = 0;
        }
    } else if (warp == 3) {
        // ===== issuer of the second product: A = residual pieces in tensor memory, B = the item's X tile (MN-major) =====
        const uint32_t x_ring_addr = smem_u32(x_ring);
        const uint32_t tmem_g = tmem_base + F_COL_G;
        int segs_done = 0;
        int n_tile = t_begin % tiles_n;
        bool first_of_seg = true;
        for (int t = t_begin, L = 0; t < t_end; ++t, ++L) {
            const bool last_of_seg = (t + 1 >= t_end) || (n_tile + 1 == tiles_n);
            const int rb = L & 1, stage = L % H_XSTAGES;
            mbar_wait(&r_full[rb], (L >> 1) & 1);
            mbar_wait(&x_full[stage], (L / H_XSTAGES) & 1);               // already complete; orders this warp after the TMA
            if (first_of_seg && segs_done > 0) mbar_wait(g_empty, (segs_done - 1) & 1);   // G drained
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint64_t xd = make_desc_mn(x_ring_addr + (uint32_t)stage * F_XSTAGE, F_XBOX, 1024);
            const uint32_t tmem_r = tmem_base + H_COL_R + (uint32_t)rb * H_RBUF_COLS;
            if (elect_one()) {
#pragma unroll
                for (int p = 0; p < 2; ++p)
#pragma unroll
                    for (int k = 0; k < FN / UMMA_K; ++k)
                        umma_bf16_ts(tmem_g, tmem_r + (uint32_t)(p * H_RPIECE_COLS + k * (UMMA_K / 2)),
                                     xd + (uint64_t)((k * UMMA_K * 128) >> 4), IDESC_G16,
                                     (first_of_seg && p == 0 && k == 0) ? 0u : 1u);
                tcgen05_commit(&x_empty[stage]);
                tcgen05_commit(&r_empty[rb]);
                if (last_of_seg) tcgen05_commit(g_full);
            }
            __syncwarp();
            first_of_seg = last_of_seg;
            if (last_of_seg) ++segs_done;
            if (++n_tile == tiles_n) n_tile = 0;
        }
    } else if (warp >= 4) {
        // ===== epilogue warps =====
        const int q = warp & 3, part = (warp - 4) >> 2;
        const int trow = q * 32 + lane;                        // row of the 128-chain tile = TMEM lane
        const int c0 = part * 16;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const float l2_scale = 1.4426950408889634f * fa.s_scale;     // accumulator -> s log2(e)
        uint32_t ra[8], rb8[8];
        // 8 accumulator columns (s * 2^20) -> 4 + 4 packed fp16 residual words; returns the potential terms.
        // Packed f32x2 arithmetic (FMUL2 / FADD2 / FFMA2 on sm_100) wherever the operation has no operand modifier;
        // special functions batched: one ex2 per element, one rcp per PAIR (1/a = b / (a b)), one lg2 per 8 elements
        // (sum of logs = log of the product; every factor is in (1, 2]).
        auto half_item = [&](const uint32_t* r, const float* y, uint32_t* q0, uint32_t* q1) -> float {
            float2 pacc;
            float2 den2[4], num2[4];
            float pp[4];
            const float2 lscale = make_float2(l2_scale, l2_scale), one2 = make_float2(1.f, 1.f);
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const float2 sv2 = make_float2(__uint_as_float(r[2 * h]), __uint_as_float(r[2 * h + 1]));
                const float2 t2 = fmul2(sv2, lscale);                    // s log2(e)
                const float2 e2 = make_float2(ex2_approx(-fabsf(t2.x)), ex2_approx(-fabsf(t2.y)));
                den2[h] = fadd2(e2, one2);
                num2[h] = make_float2(sv2.x >= 0.f ? 1.f : e2.x, sv2.y >= 0.f ? 1.f : e2.y);   // numerator of sigmoid(s)
                // |t| sums per lane, packed (FADD2 takes |.| operands); starting from the first |t| has the bits of 0 + |t|
                const float2 at2 = make_float2(fabsf(t2.x), fabsf(t2.y));
                pacc = h == 0 ? at2 : fadd2(pacc, at2);
                pp[h] = den2[h].x * den2[h].y;
            }
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const float rp = rcp_approx(pp[h]);
                const float2 inv2 = fmul2(make_float2(den2[h].y, den2[h].x), make_float2(rp, rp));
                const float2 rr = ffma2(num2[h], inv2, make_float2(-y[2 * h], -y[2 * h + 1]));     // sigmoid(s) - y
                const __half2 hi = __floats2half2_rn(rr.x, rr.y);
                const __half2 lo = __floats2half2_rn(sub_f16(rr.x, __low2half(hi)), sub_f16(rr.y, __high2half(hi)));
                q0[h] = *reinterpret_cast<const uint32_t*>(&hi);
                q1[h] = *reinterpret_cast<const uint32_t*>(&lo);
            }
            // (pp0 pp1, pp2 pp3) as one packed product
            const float2 pq = fmul2(make_float2(pp[0], pp[2]), make_float2(pp[1], pp[3]));
            const float prod = pq.x * pq.y;
            // sum of 1/2 |s| + log(1 + exp(-|s|)):  |s| = |t| ln 2
            return 0.6931471805599453f * fmaf(0.5f, pacc.x + pacc.y, lg2_approx(prod));
        };
        float urun = 0.f;
        // One work item L of a segment: S(L) -> residual pieces in tensor memory, its potential terms added to urun.
        // BUF = L & 1 is a template constant so that every tensor-memory address is an immediate off lane_addr;
        // ph = (L >> 1) & 1 is the parity of S(L)'s fill and of the previous release of residual buffer BUF.
        // On entry ra holds (or is receiving) columns [c0, c0 + 8) of S(L); with has_next the same columns of S(L + 1)
        // are requested before the second half of this item is processed.  partial is set only for the last data
        // tile when N is not a multiple of FN; lim = N - (first row of the tile) - c0.
        auto item = [&](auto bufc, uint32_t ph, const float* yp, bool has_next, bool partial, int lim) {
            constexpr uint32_t BUF = decltype(bufc)::value;
            float yv[16];
            if (!partial) {
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                    const float4 y4 = __ldg(reinterpret_cast<const float4*>(yp + j));
                    yv[j] = y4.x; yv[j + 1] = y4.y; yv[j + 2] = y4.z; yv[j + 3] = y4.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j) yv[j] = (j < lim) ? __ldg(yp + j) : 0.5f;
            }
            // The 16 accumulator columns of this thread are read as two halves so that the tensor-memory read of one
            // half (TMEM reads run at ~64 B/clk per SM: 32 KB per item) overlaps the arithmetic of the other.
            uint32_t p0[8], p1[8];
            float uacc = 0.f;
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");          // ra = columns [c0, c0 + 8) of S(L)
            tmem_ld8(lane_addr + (uint32_t)c0 + (BUF * FN + 8), rb8);
            uacc += half_item(ra, yv, p0, p1);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");          // rb8 = columns [c0 + 8, c0 + 16)
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&s_empty[BUF])) : "memory");
            if (has_next) {
                mbar_wait_backoff(&s_full[BUF ^ 1], ph ^ BUF);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                tmem_ld8(lane_addr + (uint32_t)c0 + ((BUF ^ 1) * FN), ra);
            }
            uacc += half_item(rb8, yv + 8, p0 + 4, p1 + 4);
            // rows past the end of the data (s = 0 from the zero-filled X rows, y loaded as 1/2): the residual is 0 by
            // construction and each such row added log 2 to the potential
            if (partial) uacc -= 0.6931471805599453f * (float)min(16, max(0, 16 - lim));
            urun += uacc;
            // residual pieces -> tensor memory (the second product of item L - 2 must have consumed this buffer)
            mbar_wait(&r_empty[BUF], ph ^ 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t raddr = lane_addr + (uint32_t)(part * 8) + (H_COL_R + BUF * H_RBUF_COLS);
            tmem_st8(raddr, p0);
            tmem_st8(raddr + H_RPIECE_COLS, p1);
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&r_full[BUF])) : "memory");
        };
        const std::integral_constant<uint32_t, 0> buf0;
        const std::integral_constant<uint32_t, 1> buf1;
        int segs_done = 0;
        // one pass per segment: the items of one chain tile within this CTA's range
        for (int t = t_begin, L = 0; t < t_end;) {
            const int m_tile = t / tiles_n, n_first = t - m_tile * tiles_n;
            const int cnt = min(t_end - t, tiles_n - n_first);
            {
                // beta pieces of this chain tile -> tensor memory (the first products of the previous segment retired)
                mbar_wait(a_free, (segs_done & 1) ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const int row = m_tile * BM + trow;
                if (part * 32 < KB * BK) {
#pragma unroll
                    for (int p = 0; p < 2; ++p) {
                        uint32_t bw[16];
                        const __half* src = fa.beta + (long long)p * fa.plane_stride + (long long)row * fa.dim + part * 32;
#pragma unroll
                        for (int v = 0; v < 4; ++v) {
                            uint4 w = make_uint4(0u, 0u, 0u, 0u);
                            if (row < fa.M && part * 32 + v * 8 < fa.dim) w = __ldg(reinterpret_cast<const uint4*>(src + v * 8));
                            bw[4 * v] = w.x; bw[4 * v + 1] = w.y; bw[4 * v + 2] = w.z; bw[4 * v + 3] = w.w;
                        }
                        tmem_st16(lane_addr + H_COL_B + (uint32_t)(p * H_BPIECE_COLS + part * 16), bw);
                    }
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(a_full)) : "memory");
            }
            // nothing was requested ahead for the first item (the beta pieces had to be in place first)
            mbar_wait_backoff(&s_full[L & 1], (L >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            tmem_ld8(lane_addr + (uint32_t)((L & 1) * FN + c0), ra);

            // steady state: every item but the last of the segment is a full data tile followed by one more item;
            // pairs start on an even L so that both buffer indices are constants
            const float* yp = fa.y + n_first * FN + c0;
            uint32_t ph = (L >> 1) & 1;
            int k = cnt - 1;
            if (k > 0 && (L & 1)) { item(buf1, ph, yp, true, false, FN); ph ^= 1; yp += FN; --k; }
            for (; k >= 2; k -= 2) {
                item(buf0, ph, yp, true, false, FN);
                item(buf1, ph, yp + FN, true, false, FN);
                ph ^= 1;
                yp += 2 * FN;
            }
            if (k) { item(buf0, ph, yp, true, false, FN); yp += FN; }

            // last item of the segment: nothing to request ahead; the last data tile may be partial
            const int L_last = L + cnt - 1, n_last = n_first + cnt - 1;
            const bool partial = n_last * FN + FN > fa.N;
            const int lim = fa.N - n_last * FN - c0;
            if (L_last & 1) item(buf1, (uint32_t)(L_last >> 1) & 1, yp, false, partial, lim);
            else item(buf0, (uint32_t)(L_last >> 1) & 1, yp, false, partial, lim);

            {
                // drain G: this warp's lane quadrant, columns [32 part, 32 part + 32)
                mbar_wait(g_full, segs_done & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                uint32_t gq[32];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(gq[0]), "=r"(gq[1]), "=r"(gq[2]), "=r"(gq[3]), "=r"(gq[4]), "=r"(gq[5]), "=r"(gq[6]), "=r"(gq[7]),
                      "=r"(gq[8]), "=r"(gq[9]), "=r"(gq[10]), "=r"(gq[11]), "=r"(gq[12]), "=r"(gq[13]), "=r"(gq[14]),
                      "=r"(gq[15]), "=r"(gq[16]), "=r"(gq[17]), "=r"(gq[18]), "=r"(gq[19]), "=r"(gq[20]), "=r"(gq[21]),
                      "=r"(gq[22]), "=r"(gq[23]), "=r"(gq[24]), "=r"(gq[25]), "=r"(gq[26]), "=r"(gq[27]), "=r"(gq[28]),
                      "=r"(gq[29]), "=r"(gq[30]), "=r"(gq[31])
                    : "r"(lane_addr + F_COL_G + (uint32_t)(part * 32)));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(g_empty)) : "memory");
                ++segs_done;
                const int row = m_tile * BM + trow;
                if (row < fa.M) {
                    const int b_first = (int)(((long long)m_tile * tiles_n) / fa.per_cta);
                    float* orow = fa.gpart + (long long)(blockIdx.x - b_first) * fa.plane_stride + (long long)row * fa.dim;
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const int col = part * 32 + j;
                        if (col + 3 < fa.dim) {
                            *reinterpret_cast<float4*>(orow + col) =
                                make_float4(__uint_as_float(gq[j]), __uint_as_float(gq[j + 1]), __uint_as_float(gq[j + 2]),
                                            __uint_as_float(gq[j + 3]));
                        } else {
                            for (int e = 0; e < 4; ++e)
                                if (col + e < fa.dim) orow[col + e] = __uint_as_float(gq[j + e]);
                        }
                    }
                    fa.upart[((long long)blockIdx.x * EPI_PARTS + part) * fa.M + row] = (double)urun;
                }
                urun = 0.f;
            }
            t += cnt;
            L += cnt;
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(F_TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side: tensor maps through the driver entry point (no link-time dependency on libcuda)
// ---------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return nullptr;
        fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 2D bf16 row-major [rows][cols] (cols contiguous, row pitch ld elements), box = 64 x 128, 128-byte swizzle
static int make_map(CUtensorMap* map, const void* base, long long rows, long long cols, long long ld, int box_rows = BM,
                    CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
    EncodeTiledFn enc = get_encode();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return B2H_ERR_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed: " + std::to_string((int)r)); return B2H_ERR_CUDA; }
    return 0;
}

}  // namespace tc

// out[z][M x N] (fp32, row pitch ldo, plane stride split_stride) = sum_p A[p*piece_rows + m][k] * B[n][k]
// over the k-blocks of split z.  A: [pieces*piece_rows x K] bf16 (pitch lda), B: [N x K] bf16 (pitch ldb).
static int tc_launch(cudaStream_t st, const void* A, long long lda, const void* B, long long ldb, float* out, int M, int N,
                     int K, int pieces, int piece_rows, int ldo, int nsplit, long long split_stride, tc::Epilogue ep,
                     int a_blocked = 0, int* resident_tiles_per_cta = nullptr) {
    using namespace tc;
    // checked before anything is launched: a split plane stride that is not a multiple of four floats misaligns the
    // epilogue's float4 stores, and a short pitch or piece makes the TMA boxes read another row's (or piece's) data
    if (M < 1 || N < 1 || K < 1 || pieces < 1 || piece_rows < M) {
        set_error("tc_gemm: M, N, K and pieces must be positive and piece_rows >= M");
        return B2H_ERR_ARG;
    }
    const bool short_a = a_blocked ? (long long)piece_rows < (long long)((K + BN - 1) / BN) * ((M + BM - 1) / BM) * BM
                                   : lda < K;
    if (short_a || ldb < K) { set_error("tc_gemm: the A or B rows do not hold K elements"); return B2H_ERR_ARG; }
    if (ep.mode == 0 && ldo < N) { set_error("tc_gemm: ldo must be >= N"); return B2H_ERR_ARG; }
    if (ep.mode == 0 && nsplit > 1 && (split_stride % 4 || split_stride < (long long)(M - 1) * ldo + N)) {
        set_error("tc_gemm: split_stride must be a multiple of 4 and hold an M x N plane");
        return B2H_ERR_ARG;
    }
    if ((lda * 2) % 16 || (ldb * 2) % 16 || ((uintptr_t)A & 15) || ((uintptr_t)B & 15) || ((uintptr_t)out & 15) || ldo % 4) {
        set_error("tc_gemm: operands must be 16-byte aligned with 16-byte row pitches");
        return B2H_ERR_ARG;
    }
    CUtensorMap ma, mb;
    // blocked A: a 2D view [pieces * piece_rows][128] with a 128-element pitch (piece_rows counts blocked rows)
    int rc = a_blocked ? make_map(&ma, A, (long long)pieces * piece_rows, BN, BN)
                       : make_map(&ma, A, (long long)pieces * piece_rows, K, lda);
    if (rc) return rc;
    rc = make_map(&mb, B, N, K, ldb);
    if (rc) return rc;
    const int kb_total = (K + BK - 1) / BK;
    if (nsplit < 1) nsplit = 1;
    if (nsplit > kb_total) nsplit = kb_total;
    const int kb_per = (kb_total + nsplit - 1) / nsplit;
    nsplit = (kb_total + kb_per - 1) / kb_per;
    const int tiles_n = (N + BN - 1) / BN, tiles_m = (M + BM - 1) / BM;
    static int sm_count = 0;
    if (!sm_count) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
        if (sm_count <= 0) sm_count = 148;
    }
    const long long total = (long long)tiles_n * tiles_m * nsplit;
    if (!a_blocked && nsplit == 1 && pieces * kb_total <= RES_A_BLOCKS && kb_total <= RES_KB && total >= 2 * sm_count) {
        // short reduction, many column tiles: keep A resident, stream B once per tile
        const int per = (int)((total + sm_count - 1) / sm_count);
        const int grid_r = (int)((total + per - 1) / per);
        B2H_CUDA(cudaFuncSetAttribute(tc_gemm_resident_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RES_SMEM));
        tc_gemm_resident_kernel<<<grid_r, THREADS, RES_SMEM, st>>>(ma, mb, out, M, N, K, pieces, piece_rows, ldo, tiles_m,
                                                                   tiles_n, per, ep);
        B2H_LAUNCH_CHECK();
        if (resident_tiles_per_cta) *resident_tiles_per_cta = per;
        return 1;
    }
    if (resident_tiles_per_cta) *resident_tiles_per_cta = 0;
    const int grid = (int)std::min<long long>(total, sm_count);
    // short reductions (the S product: K = dim) take a shallow ring so that three CTAs share an SM and one CTA's
    // epilogue overlaps the others' loads and MMAs; long reductions take the full 6-stage ring
    const int iters = kb_per * pieces;
    const int stages = STAGES;
    (void)iters;
    B2H_CUDA(cudaFuncSetAttribute(tc_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(STAGES)));
    tc_gemm_kernel<<<grid, THREADS, smem_bytes(stages), st>>>(ma, mb, out, M, N, K, pieces, piece_rows, ldo, kb_per,
                                                             split_stride, stages, tiles_m, tiles_n, nsplit, a_blocked, ep);
    B2H_LAUNCH_CHECK();
    return nsplit;
}

int tc_gemm(cudaStream_t st, const void* A, long long lda, const void* B, long long ldb, float* out, int M, int N, int K,
            int pieces, int piece_rows, int ldo, int nsplit, long long split_stride) {
    tc::Epilogue ep{0, nullptr, nullptr, 0, 0, nullptr};
    return tc_launch(st, A, lda, B, ldb, out, M, N, K, pieces, piece_rows, ldo, nsplit, split_stride, ep, 0);
}

// S = sum_p A_p . B^T never leaves the SM: the epilogue writes the residual pieces (bf16, tile-blocked:
// [3][ceil(N/128)][ceil(M/128)][128][128]) and the per-tile partial sums of the potential, upart[4 * ceil(N/128)][M].
// *tiles_per_cta > 0: upart is [CTA][4][M] (each CTA covers tiles_per_cta consecutive tiles, column tile fastest);
// otherwise upart is [column tile][4][M].
int tc_gemm_logistic(cudaStream_t st, const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
                     int pieces, int piece_rows, const float* y, void* R, long long r_piece_stride, double* upart,
                     int* tiles_per_cta) {
    if (((uintptr_t)R & 1023)) { set_error("tc_gemm_logistic: residual buffer must be 1024-byte aligned"); return B2H_ERR_ARG; }
    tc::Epilogue ep{1, y, (__nv_bfloat16*)R, r_piece_stride, (M + tc::BM - 1) / tc::BM, upart};
    return tc_launch(st, A, lda, B, ldb, nullptr, M, N, K, pieces, piece_rows, 4, 1, 0, ep, 0, tiles_per_cta);
}

// out[z] = sum_p R_p . B^T with R in the tile-blocked layout written by tc_gemm_logistic (K = data rows).
int tc_gemm_blocked_a(cudaStream_t st, const void* R, long long r_piece_stride, const void* B, long long ldb, float* out,
                      int M, int N, int K, int pieces, int ldo, int nsplit, long long split_stride) {
    tc::Epilogue ep{0, nullptr, nullptr, 0, 0, nullptr};
    const int piece_rows = (int)(r_piece_stride / tc::BN);
    return tc_launch(st, R, tc::BN, B, ldb, out, M, N, K, pieces, piece_rows, ldo, nsplit, split_stride, ep, 1);
}


// Fully fused gradient: see tc_logistic_fused_kernel.  beta_pieces: [3 * piece_rows x dim] bf16, X: [N x dim] bf16.
// Writes gpart[plane][M x dim] (fp32) and upart[CTA][4][M]; *per_cta = items per CTA, *planes = planes a chain
// tile can receive (the reduction kernels recompute which CTAs touched a tile from per_cta).
int tc_logistic_fused(cudaStream_t st, const void* beta_pieces, int piece_rows, const void* X, int M, int N, int dim,
                      const float* y, float* gpart, double* upart, int* per_cta, int* planes) {
    using namespace tc;
    if (dim > 2 * BK || dim % 8) { set_error("tc_logistic_fused: dim must be a multiple of 8, at most 128"); return B2H_ERR_ARG; }
    CUtensorMap mb, mx;
    int rc = make_map(&mb, beta_pieces, 3ll * piece_rows, dim, dim);
    if (rc) return rc;
    rc = make_map(&mx, X, N, dim, dim, FN);
    if (rc) return rc;
    static int sm_count = 0;
    if (!sm_count) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
        if (sm_count <= 0) sm_count = 148;
    }
    FusedArgs fa;
    fa.y = y; fa.gpart = gpart; fa.plane_stride = (long long)M * dim; fa.upart = upart;
    fa.M = M; fa.N = N; fa.dim = dim; fa.piece_rows = piece_rows;
    fa.tiles_m = (M + BM - 1) / BM;
    fa.tiles_n = (N + FN - 1) / FN;
    const long long total = (long long)fa.tiles_m * fa.tiles_n;
    fa.per_cta = (int)((total + sm_count - 1) / sm_count);
    const int grid = (int)((total + fa.per_cta - 1) / fa.per_cta);
    auto launch = [&](auto kern) -> int {
        B2H_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F_SMEM));
        kern<<<grid, THREADS, F_SMEM, st>>>(mb, mx, fa);
        return 0;
    };
    rc = dim > BK ? launch(tc_logistic_fused_kernel<2>) : launch(tc_logistic_fused_kernel<1>);
    if (rc) return rc;
    B2H_LAUNCH_CHECK();
    *per_cta = fa.per_cta;
    *planes = logistic_fused_planes(M, N);
    return 0;
}

// fp16 x 2 fused gradient: see tc_logistic_fused16_kernel.  beta_pieces: [2][M x dim] fp16 (beta * 2^(acc_exp - shift)),
// X16: [N x dim] fp16 = X * 2^shift.  gpart comes out scaled by 2^shift; the potential partials lack the part
// that is linear in beta (see the kernel).
int tc_logistic_fused16(cudaStream_t st, const void* beta_pieces, const void* X16, int acc_exp, int M, int N, int dim,
                        const float* y, float* gpart, double* upart, int* per_cta) {
    using namespace tc;
    if (dim > 2 * BK || dim % 8) { set_error("tc_logistic_fused16: dim must be a multiple of 8, at most 128"); return B2H_ERR_ARG; }
    CUtensorMap mx;
    int rc = make_map(&mx, X16, N, dim, dim, FN, CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    if (rc) return rc;
    static int sm_count = 0;
    if (!sm_count) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
        if (sm_count <= 0) sm_count = 148;
    }
    Fused16Args fa;
    fa.y = y; fa.beta = (const __half*)beta_pieces; fa.gpart = gpart; fa.plane_stride = (long long)M * dim;
    fa.upart = upart; fa.s_scale = ldexpf(1.f, -acc_exp);
    fa.M = M; fa.N = N; fa.dim = dim;
    fa.tiles_m = (M + BM - 1) / BM;
    fa.tiles_n = (N + FN - 1) / FN;
    const long long total = (long long)fa.tiles_m * fa.tiles_n;
    fa.per_cta = (int)((total + sm_count - 1) / sm_count);
    const int grid = (int)((total + fa.per_cta - 1) / fa.per_cta);
    if (dim > BK) {
        B2H_CUDA(cudaFuncSetAttribute(tc_logistic_fused16_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)H_SMEM));
        tc_logistic_fused16_kernel<2><<<grid, THREADS, H_SMEM, st>>>(mx, fa);
    } else {
        B2H_CUDA(cudaFuncSetAttribute(tc_logistic_fused16_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)H_SMEM));
        tc_logistic_fused16_kernel<1><<<grid, THREADS, H_SMEM, st>>>(mx, fa);
    }
    B2H_LAUNCH_CHECK();
    *per_cta = fa.per_cta;
    return 0;
}

// upper bound on the number of CTAs whose item range intersects one chain tile
int logistic_fused_planes(int M, int N) {
    const long long tiles_m = (M + tc::BM - 1) / tc::BM, tiles_n = (N + tc::FN - 1) / tc::FN;
    int sm_count = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (sm_count <= 0) sm_count = 148;
    const long long per = (tiles_m * tiles_n + sm_count - 1) / sm_count;
    return (int)((tiles_n + per - 1) / per + 1);
}

}  // namespace b2h

// the kernels index with int: sizes above INT_MAX would wrap
static bool ints_fit(std::initializer_list<int64_t> v) {
    for (int64_t x : v)
        if (x < 0 || x > 0x7fffffff) { b2h::set_error("tc_gemm: size out of range"); return false; }
    return true;
}

extern "C" int b2h_tc_gemm_bf16(b2h_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, float* out, int64_t M,
                                int64_t N, int64_t K, int32_t pieces, int64_t piece_rows, int64_t ldo, int32_t nsplit,
                                int64_t split_stride) {
    if (!ctx) { b2h::set_error("null context"); return B2H_ERR_ARG; }
    // the TMA row coordinate of the last piece, p * piece_rows + row, is an int as well
    if (!ints_fit({M, N, K, piece_rows, ldo}) || !ints_fit({(int64_t)pieces * piece_rows})) return B2H_ERR_ARG;
    int rc = b2h::tc_gemm(ctx->stream, A, lda, B, ldb, out, (int)M, (int)N, (int)K, pieces, (int)piece_rows, (int)ldo,
                          nsplit, split_stride);
    return rc < 0 ? rc : 0;
}

extern "C" int b2h_tc_logistic_residual(b2h_ctx* ctx, const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M,
                                        int64_t N, int64_t K, int32_t pieces, int64_t piece_rows, const float* y, void* R,
                                        int64_t r_piece_stride, double* upart, int32_t* tiles_per_cta) {
    if (!ctx || !y || !R || !upart || !tiles_per_cta) { b2h::set_error("null argument"); return B2H_ERR_ARG; }
    if (!ints_fit({M, N, K, piece_rows}) || !ints_fit({(int64_t)pieces * piece_rows})) return B2H_ERR_ARG;
    const int64_t tile_elems = (int64_t)b2h::tc::BM * b2h::tc::BN;
    if (M > 0 && N > 0 && r_piece_stride < (N + b2h::tc::BN - 1) / b2h::tc::BN * ((M + b2h::tc::BM - 1) / b2h::tc::BM) * tile_elems) {
        b2h::set_error("tc_logistic_residual: r_piece_stride does not hold the tile-blocked M x N residual");
        return B2H_ERR_ARG;
    }
    if (r_piece_stride % 8 || ((uintptr_t)y & 15)) {     // 16-byte stores of the pieces, 16-byte loads of y
        b2h::set_error("tc_logistic_residual: r_piece_stride must be a multiple of 8 and y 16-byte aligned");
        return B2H_ERR_ARG;
    }
    int per = 0;
    int rc = b2h::tc_gemm_logistic(ctx->stream, A, lda, B, ldb, (int)M, (int)N, (int)K, pieces, (int)piece_rows, y, R,
                                   r_piece_stride, upart, &per);
    if (rc < 0) return rc;
    *tiles_per_cta = per;
    return 0;
}

extern "C" int b2h_tc_gemm_blocked_bf16(b2h_ctx* ctx, const void* R, int64_t r_piece_stride, const void* B, int64_t ldb,
                                        float* out, int64_t M, int64_t N, int64_t K, int32_t pieces, int64_t ldo,
                                        int32_t nsplit, int64_t split_stride) {
    if (!ctx) { b2h::set_error("null context"); return B2H_ERR_ARG; }
    if (!ints_fit({M, N, K, ldo, r_piece_stride / b2h::tc::BN}) || !ints_fit({(int64_t)pieces * (r_piece_stride / b2h::tc::BN)}))
        return B2H_ERR_ARG;
    if (r_piece_stride % b2h::tc::BN) { b2h::set_error("tc_gemm_blocked: r_piece_stride must be a multiple of 128"); return B2H_ERR_ARG; }
    int rc = b2h::tc_gemm_blocked_a(ctx->stream, R, r_piece_stride, B, ldb, out, (int)M, (int)N, (int)K, pieces, (int)ldo,
                                    nsplit, split_stride);
    return rc < 0 ? rc : 0;
}
