// Host-side declarations shared by the translation units of libb200hmc.so.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/b200hmc.h"

struct b2h_ctx {
    int device;
    cudaStream_t stream;
    int sm_count;
    // side stream for the dense-metric momentum contractions (a few row tiles per tick): run beside the main
    // stream's kernels they share SMs fluidly instead of adding a mostly empty wave to a full launch
    cudaStream_t side;
    cudaEvent_t ev_pre[2], ev_side[2];
    // dense-metric runs of the split engine hop from the caller's stream onto this high-priority stream (and back at
    // the end of the call), so that the side stream's momentum tiles -- lowest priority -- only take SMs no full-size
    // launch is waiting for (the 8 of 148 a 288-tile contraction leaves idle in its second wave)
    cudaStream_t hi;
    cudaEvent_t ev_hop;
    int* host_flag;   // pinned, for the split engine's completion poll
    // b2h_tick_timer: event pairs around the tick-kernel launches of the split engine (measurement aid, off by default)
    int tick_timer = 0;               // 0 off, 1 the tick kernel, 2 the gradient call (potential_and_grad) of every tick
    std::vector<cudaEvent_t> tick_events;
    size_t tick_events_used = 0;
    double tick_ms = 0.0;
    long long tick_launches = 0;
};

namespace b2h {

typedef long long i64;

void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);

#define B2H_CUDA(expr)                                        \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) return ::b2h::cuda_fail(_e, #expr); \
    } while (0)

#define B2H_LAUNCH_CHECK() B2H_CUDA(cudaGetLastError())

// gemm.cu
template <typename T>
struct GemmGroup {
    const T* A; i64 lda;
    const T* B; i64 ldb;
    T* out; i64 ldo;
    int M;                 // rows (upper bound when m_dev is given)
    const int* m_dev;      // optional device-side row count
    const T* sub;          // optional [K] vector subtracted from every A row on load
    const int* in_rows;    // optional gather list: A row of logical row r is in_rows[r]
    const int* out_rows;   // optional scatter list for the output rows
    int tri;               // B known to be 1: upper-triangular (B[k][n] = 0 for k > n), 2: lower-triangular, 0: general.
                           // The DMMA tile kernel then skips the k-range of a column tile that only holds zeros.
};
template <typename T>
void launch_gemm_grouped(cudaStream_t st, const GemmGroup<T>& g0, const GemmGroup<T>& g1, const GemmGroup<T>& g2, int N,
                         int K, int nsplit, i64 split_stride, int rider_tile_rows);

template <typename T>
void launch_dense_apply(cudaStream_t st, const T* A, const T* B, T* out, int M, int N, int K, const int* m_dev,
                        const T* sub);

// dense_per_chain.cu: out[m][chain(r)] = in[r] . M[m][chain(r)] for rows r < min(rows, *count), chain(r) = list[r]
// (identity when list is null); M[m] + c * d * d is chain c's [d x d] matrix, tri[m] as GemmGroup::tri.  One matrix
// (M[1] = nullptr) or two from the same input row (the momentum rider).
template <typename T>
struct PcJob {
    const T* in;
    const T* M[2];
    T* out[2];
    int tri[2];
    const int* count;      // optional device-side row count
    const int* list;       // optional row -> chain list
    i64 rows;
    int d;
};
template <typename T>
void launch_dense_pc(cudaStream_t st, const PcJob<T>& job);
template <typename T>
void launch_dense_apply_pc(cudaStream_t st, const T* in, const T* M, T* out, i64 C, int d, int tri);

template <typename T>
void launch_gemm(cudaStream_t st, const T* A, i64 lda, const T* B, i64 ldb, T* out, i64 ldo, int M, int N, int K,
                 const int* m_dev, const T* sub, int nsplit, i64 split_stride);

// primitives.cu
template <typename T>
int potential_and_grad_impl(b2h_ctx* ctx, const b2h_model* m, const T* q, T* U, T* g, i64 C, void* ws, i64 ws_bytes,
                            bool gradient_only = false);   // gradient_only: the caller forms U itself (EngineView::u_center)
i64 potential_workspace_bytes_impl(const b2h_model* m, int dtype, i64 C);

// logreg.cu
template <typename T>
int logistic_potential_and_grad(b2h_ctx* ctx, const b2h_model* m, const T* q, T* U, T* g, i64 C, void* ws,
                                i64 ws_bytes, int path);
i64 logistic_workspace_bytes(const b2h_model* m, int dtype, i64 C);

// tc_gemm.cu (tcgen05 / TMA); returns the number of split-K planes written, or < 0
int tc_gemm(cudaStream_t st, const void* A, long long lda, const void* B, long long ldb, float* out, int M, int N, int K,
            int pieces, int piece_rows, int ldo, int nsplit, long long split_stride);

int tc_gemm_logistic(cudaStream_t st, const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
                     int pieces, int piece_rows, const float* y, void* R, long long r_piece_stride, double* upart,
                     int* tiles_per_cta);
int tc_gemm_blocked_a(cudaStream_t st, const void* R, long long r_piece_stride, const void* B, long long ldb, float* out,
                      int M, int N, int K, int pieces, int ldo, int nsplit, long long split_stride);

int tc_logistic_fused(cudaStream_t st, const void* beta_pieces, int piece_rows, const void* X, int M, int N, int dim,
                      const float* y, float* gpart, double* upart, int* per_cta, int* planes);
int logistic_fused_planes(int M, int N);
int tc_logistic_fused16(cudaStream_t st, const void* beta_pieces, const void* X16, int acc_exp, int M, int N, int dim,
                        const float* y, float* gpart, double* upart, int* per_cta);

// user_model.cu (NVRTC-compiled user log-density, thread per chain)
template <typename T>
int user_potential_and_grad(b2h_ctx* ctx, const b2h_model* m, const T* q, T* U, T* g, i64 C, void* ws, i64 ws_bytes);
i64 user_workspace_bytes(const b2h_model* m, int dtype, i64 C);

// engine_kernels.cu
int nuts_run_impl(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                  const b2h_cfg* cfg, const b2h_adapt* adapt, void* q, void* p, void* U, void* g, double* step_size,
                  i64 C, int n_transitions, i64 max_ticks, int resume, b2h_diag* diag, void* draws,
                  double* draw_stats, int n_store, int64_t* counters, void* ws, i64 ws_bytes, bool hmc);
int nuts_expand_impl(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                     const b2h_cfg* cfg, b2h_tree* tree, const double* eps, i64 C, b2h_diag* diag, void* ws, i64 ws_bytes);
int nuts_subtree_impl(b2h_ctx* ctx, const b2h_model* model, const b2h_metric* metric, const b2h_rng* rng,
                      const b2h_cfg* cfg, b2h_subtree* sub, const double* eps, i64 C, void* ws, i64 ws_bytes);
i64 engine_workspace_bytes(const b2h_model* model, const b2h_metric* metric, const b2h_cfg* cfg, i64 C);
int engine_plan_group(const b2h_model* model, const b2h_metric* metric, const b2h_cfg* cfg, i64 C, bool free_running);

static inline size_t dtype_size(int dtype) { return dtype == B2H_F64 ? 8 : 4; }

}  // namespace b2h
