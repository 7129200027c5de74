// Shared between the engine translation units (engine_kernels.cu: workspace, entry points;
// engine_fused_*.cu: the persistent kernel; engine_split_*.cu: the per-tick kernels).  One TU per element
// type keeps the build parallel.
#pragma once

#include "engine.cuh"
#include "launch.h"

namespace b2h {

constexpr int kRiderSplit = 5;      // split-K slices of the momentum contractions (few rows, full K)

struct EnginePlan {
    int G;
    bool dense, split, hmc, per_chain_imm, scalar_imm;
    bool dense_per_chain;   // B2H_IMM_DENSE_PER_CHAIN: dense (same tick kernels), the metric mat-vecs per chain
    size_t model_ws_off, model_ws_bytes;
};

// ---------------------------------------------------------------------------
// fused persistent kernel
// ---------------------------------------------------------------------------
template <int G>
struct Geo {
    static constexpr int kThreads = G > 32 ? G : 128;
    static constexpr int kChainsPerBlock = G > 32 ? 1 : 128 / G;
    // the per-tick (split) kernels are latency-bound streams: cap registers at 64 for 50% occupancy
    static constexpr int kMinBlocksSplit = G > 32 ? 4 : 8;
    // post + pre of consecutive ticks with the front in registers (split_postpre_kernel)
#ifndef B2H_TICK_MINB
#define B2H_TICK_MINB 2
#endif
    static constexpr int kMinBlocksTick = G > 32 ? B2H_TICK_MINB : 2 * B2H_TICK_MINB;
    // the persistent fused kernel is latency / instruction-fetch bound: favour resident warps over registers
    static constexpr int kMinBlocksFused = G > 32 ? 3 : 5;
    __device__ static int chain() {
        return G > 32 ? (int)blockIdx.x : (int)(blockIdx.x * kChainsPerBlock + threadIdx.x / G);
    }
    static int grid(int C) { return (C + kChainsPerBlock - 1) / kChainsPerBlock; }
};

// E > 0: the integration front stays in registers (E elements per lane) between sub-tree boundaries.
template <typename T, int E> struct FrontOf { typedef RegFront<T, E> type; };
template <typename T> struct FrontOf<T, 0> { typedef MemFront<T> type; };

// persistent fused kernel of every chain (engine_fused.inl); G in {1, 8, 32, 256}
template <typename T>
int launch_fused_g(cudaStream_t st, const EngineView<T>& v, const b2h_model* model, i64 max_ticks, int G, bool hmc);

// per-tick engine around the gradient / metric contractions (engine_split.inl); G in {8, 32, 256}
template <typename T>
int run_split_g(b2h_ctx* ctx, EngineView<T>& v, const EnginePlan& pl, const b2h_model* model, const b2h_metric* metric,
                const b2h_cfg* cfg, i64 max_ticks, int n_transitions, void* model_ws, i64 model_ws_bytes,
                int* not_done_dev, int resume, bool hmc);

}  // namespace b2h
