// User-supplied log-densities (SURVEY.md section 8f, row 3): the reference takes an arbitrary Python `logprob_fn` and
// differentiates it with aesara.grad (reference hmc.py:33-34, integrators.py:23); device code needs the gradient as
// device code, so the user writes ONE CUDA C++ function
//
//     template <typename T>
//     __device__ T potential_and_grad(const T* q, T* g, int d, const T* data);      // returns U(q), writes dU/dq
//
// which is compiled at run time with NVRTC for sm_100a and wrapped in a thread-per-chain kernel.  The model runs in
// the engine's split mode (one gradient launch per tick).  NVRTC is opened with dlopen: the library has no link-time
// dependency on it and b2h_user_model_create fails loudly when it is missing.
#include <dlfcn.h>

#include <string>
#include <vector>

#include "common.cuh"
#include "launch.h"

struct b2h_user_model {
    cudaLibrary_t lib;
    cudaKernel_t k32, k64;
    // reverse mode only: tape capacity in nodes per chain, and the largest count a chain needed since the last read
    // (device memory of `device`)
    bool reverse = false;
    int dim = 0;
    int device = -1;
    int64_t tape_nodes = 0;
    long long* needed = nullptr;
};

namespace b2h {

namespace {

typedef struct _nvrtcProgram* nvrtcProgram;
struct Nvrtc {
    int (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*);
    int (*CompileProgram)(nvrtcProgram, int, const char* const*);
    int (*GetProgramLogSize)(nvrtcProgram, size_t*);
    int (*GetProgramLog)(nvrtcProgram, char*);
    int (*GetCUBINSize)(nvrtcProgram, size_t*);
    int (*GetCUBIN)(nvrtcProgram, char*);
    int (*DestroyProgram)(nvrtcProgram*);
    bool ok = false;
};

Nvrtc& nvrtc() {
    static Nvrtc n;
    static bool tried = false;
    if (tried) return n;
    tried = true;
    const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12",
                           "/usr/local/cuda/lib64/libnvrtc.so"};
    void* h = nullptr;
    for (const char* nm : names)
        if ((h = dlopen(nm, RTLD_NOW | RTLD_LOCAL))) break;
    if (!h) return n;
#define B2H_SYM(field, name) *(void**)(&n.field) = dlsym(h, name); if (!n.field) return n;
    B2H_SYM(CreateProgram, "nvrtcCreateProgram")
    B2H_SYM(CompileProgram, "nvrtcCompileProgram")
    B2H_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
    B2H_SYM(GetProgramLog, "nvrtcGetProgramLog")
    B2H_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
    B2H_SYM(GetCUBIN, "nvrtcGetCUBIN")
    B2H_SYM(DestroyProgram, "nvrtcDestroyProgram")
#undef B2H_SYM
    n.ok = true;
    return n;
}

// Automatic differentiation for user densities: the user writes only
//     template <typename S, typename T> __device__ S log_density(const S* q, int d, const T* data);
// with the overloaded arithmetic below, and one of two headers supplies S:
//  - forward mode (b2h_user_model_create_ad): S = Dual<T, B2H_AD_DIM> carries the value and all d partials, so one
//    evaluation yields logprob and its gradient at O(d) per operation (small models);
//  - reverse mode (b2h_user_model_create_rev): S = Var<T> is a value and a node id; every operation on live nodes
//    appends one entry to a per-chain tape, and one reverse sweep over the tape gives the gradient at O(1) per
//    operation whatever d is.
// Both compute every value with the same expression, so U is bit-identical in the two modes.  The unary functions
// are written once (kUnary) on top of chain1(a, f, df), which each header defines for its type.  This is the role
// aesara.grad plays for the reference's logprob_fn (hmc.py:33-34).
const char* kUnary = R"(
B2H_TN B2H_D exp(const B2H_D& a) { const T e = exp(a.v); return chain1(a, e, e); }
B2H_TN B2H_D log(const B2H_D& a) { return chain1(a, log(a.v), (T)1 / a.v); }
B2H_TN B2H_D log1p(const B2H_D& a) { return chain1(a, log1p(a.v), (T)1 / ((T)1 + a.v)); }
B2H_TN B2H_D sqrt(const B2H_D& a) { const T s = sqrt(a.v); return chain1(a, s, (T)0.5 / s); }
B2H_TN B2H_D tanh(const B2H_D& a) { const T t = tanh(a.v); return chain1(a, t, (T)1 - t * t); }
B2H_TN B2H_D sin(const B2H_D& a) { return chain1(a, sin(a.v), cos(a.v)); }
B2H_TN B2H_D cos(const B2H_D& a) { return chain1(a, cos(a.v), -sin(a.v)); }
B2H_TN B2H_D square(const B2H_D& a) { return chain1(a, a.v * a.v, (T)2 * a.v); }
B2H_TN B2H_D pow(const B2H_D& a, T p) { const T f = pow(a.v, p); return chain1(a, f, p * f / a.v); }
B2H_TN B2H_D softplus(const B2H_D& a) {       // log(1 + exp(x)), stable
    const T e = exp(-fabs(a.v));
    return chain1(a, fmax(a.v, (T)0) + log1p(e), a.v >= (T)0 ? (T)1 / ((T)1 + e) : e / ((T)1 + e));
}
#undef B2H_D
#undef B2H_TN
)";

const char* kDualHeader = R"(
template <typename T, int N>
struct Dual {
    T v;
    T g[N];
    __device__ Dual() : v(0) { for (int i = 0; i < N; ++i) g[i] = 0; }
    __device__ Dual(T x) : v(x) { for (int i = 0; i < N; ++i) g[i] = 0; }
    __device__ Dual(double x, int) : v((T)x) { for (int i = 0; i < N; ++i) g[i] = 0; }
};
#define B2H_D Dual<T, N>
#define B2H_TN template <typename T, int N> __device__ inline
B2H_TN B2H_D operator+(const B2H_D& a, const B2H_D& b) { B2H_D r; r.v = a.v + b.v; for (int i = 0; i < N; ++i) r.g[i] = a.g[i] + b.g[i]; return r; }
B2H_TN B2H_D operator-(const B2H_D& a, const B2H_D& b) { B2H_D r; r.v = a.v - b.v; for (int i = 0; i < N; ++i) r.g[i] = a.g[i] - b.g[i]; return r; }
B2H_TN B2H_D operator*(const B2H_D& a, const B2H_D& b) { B2H_D r; r.v = a.v * b.v; for (int i = 0; i < N; ++i) r.g[i] = a.g[i] * b.v + a.v * b.g[i]; return r; }
B2H_TN B2H_D operator/(const B2H_D& a, const B2H_D& b) { B2H_D r; const T ib = (T)1 / b.v; r.v = a.v * ib; for (int i = 0; i < N; ++i) r.g[i] = (a.g[i] - r.v * b.g[i]) * ib; return r; }
B2H_TN B2H_D operator-(const B2H_D& a) { B2H_D r; r.v = -a.v; for (int i = 0; i < N; ++i) r.g[i] = -a.g[i]; return r; }
B2H_TN B2H_D operator+(const B2H_D& a, T b) { B2H_D r = a; r.v += b; return r; }
B2H_TN B2H_D operator+(T a, const B2H_D& b) { return b + a; }
B2H_TN B2H_D operator-(const B2H_D& a, T b) { B2H_D r = a; r.v -= b; return r; }
B2H_TN B2H_D operator-(T a, const B2H_D& b) { return (-b) + a; }
B2H_TN B2H_D operator*(const B2H_D& a, T b) { B2H_D r; r.v = a.v * b; for (int i = 0; i < N; ++i) r.g[i] = a.g[i] * b; return r; }
B2H_TN B2H_D operator*(T a, const B2H_D& b) { return b * a; }
B2H_TN B2H_D operator/(const B2H_D& a, T b) { return a * ((T)1 / b); }
B2H_TN B2H_D operator/(T a, const B2H_D& b) { return B2H_D(a) / b; }
B2H_TN B2H_D& operator+=(B2H_D& a, const B2H_D& b) { a = a + b; return a; }
B2H_TN B2H_D& operator-=(B2H_D& a, const B2H_D& b) { a = a - b; return a; }
B2H_TN B2H_D& operator+=(B2H_D& a, T b) { a.v += b; return a; }
B2H_TN B2H_D& operator-=(B2H_D& a, T b) { a.v -= b; return a; }
B2H_TN B2H_D chain1(const B2H_D& a, T f, T df) { B2H_D r; r.v = f; for (int i = 0; i < N; ++i) r.g[i] = df * a.g[i]; return r; }
)";

const char* kDualWrapper = R"(
template <typename T>
__device__ T potential_and_grad(const T* q, T* g, int d, const T* data) {
    typedef Dual<T, B2H_AD_DIM> S;
    S x[B2H_AD_DIM];
    for (int i = 0; i < d; ++i) { x[i].v = q[i]; x[i].g[i] = (T)1; }
    const S lp = log_density<S, T>(x, d, data);
    for (int i = 0; i < d; ++i) g[i] = -lp.g[i];
    return -lp.v;
}
)";

// Reverse mode.  Node ids 0..d-1 are the inputs, id d + k is the chain's k-th recorded operation, -1 a constant.
// The tape lives in the caller's workspace as five arrays, entry (row r, chain c) at r * pitch + c with
// pitch = C rounded up to 32, so a warp's 32 chains touch 32 consecutive entries:
//     id0, id1 [cap rows] int32     operand node ids (-1: none)
//     pa0, pa1 [cap rows] T         partials of the node with respect to its operands
//     adj      [d + cap rows] T     adjoints of the inputs, then of the nodes
// Operators are free functions, so the tape reaches them through block-shared state that the kernel fills from its
// parameters (two launches with different C may run at once; nothing is module-global).  The kernel's block size is
// B2H_TAPE_THREADS.  A chain that needs more than cap nodes keeps computing values, stops recording, and returns
// U = +inf, g = 0; the largest count any chain needed is atomicMax'ed into *needed.
const char* kVarHeader = R"(
#define B2H_REVERSE 1
#define B2H_TAPE_THREADS 128
struct B2hTape {
    int* id0; int* id1; void* pa0; void* pa1; void* adj;
    long long pitch;
    int cap;
    long long* needed;
};
__shared__ B2hTape b2h_tape;
__shared__ int b2h_tape_count[B2H_TAPE_THREADS];

__device__ inline long long b2h_chain() { return (long long)blockIdx.x * B2H_TAPE_THREADS + threadIdx.x; }

// records node (i0, p0, i1, p1) of this thread's chain and returns its id
template <typename T>
__device__ inline int b2h_record(int i0, T p0, int i1, T p1) {
    const int k = b2h_tape_count[threadIdx.x]++;
    if (k < b2h_tape.cap) {
        const long long e = (long long)k * b2h_tape.pitch + b2h_chain();
        b2h_tape.id0[e] = i0; b2h_tape.id1[e] = i1;
        ((T*)b2h_tape.pa0)[e] = p0; ((T*)b2h_tape.pa1)[e] = p1;
        ((T*)b2h_tape.adj)[(long long)(B2H_AD_DIM + k) * b2h_tape.pitch + b2h_chain()] = (T)0;
    }
    return B2H_AD_DIM + k;
}

template <typename T>
struct Var {
    T v;
    int id;
    __device__ Var() : v(0), id(-1) {}
    __device__ Var(T x) : v(x), id(-1) {}
    __device__ Var(double x, int) : v((T)x), id(-1) {}
};
template <typename T> __device__ inline Var<T> b2h_node(T v, int i0, T p0, int i1, T p1) {
    Var<T> r(v);
    if (i0 >= 0 || i1 >= 0) r.id = b2h_record<T>(i0, p0, i1, p1);
    return r;
}
#define B2H_D Var<T>
#define B2H_TN template <typename T> __device__ inline
B2H_TN B2H_D operator+(const B2H_D& a, const B2H_D& b) { return b2h_node(a.v + b.v, a.id, (T)1, b.id, (T)1); }
B2H_TN B2H_D operator-(const B2H_D& a, const B2H_D& b) { return b2h_node(a.v - b.v, a.id, (T)1, b.id, (T)-1); }
B2H_TN B2H_D operator*(const B2H_D& a, const B2H_D& b) { return b2h_node(a.v * b.v, a.id, b.v, b.id, a.v); }
B2H_TN B2H_D operator/(const B2H_D& a, const B2H_D& b) { const T ib = (T)1 / b.v; const T r = a.v * ib; return b2h_node(r, a.id, ib, b.id, -r * ib); }
B2H_TN B2H_D operator-(const B2H_D& a) { return b2h_node(-a.v, a.id, (T)-1, -1, (T)0); }
// adding a constant has derivative 1: the result aliases the operand's node
B2H_TN B2H_D operator+(const B2H_D& a, T b) { B2H_D r = a; r.v += b; return r; }
B2H_TN B2H_D operator+(T a, const B2H_D& b) { return b + a; }
B2H_TN B2H_D operator-(const B2H_D& a, T b) { B2H_D r = a; r.v -= b; return r; }
B2H_TN B2H_D operator-(T a, const B2H_D& b) { return (-b) + a; }
B2H_TN B2H_D operator*(const B2H_D& a, T b) { return b2h_node(a.v * b, a.id, b, -1, (T)0); }
B2H_TN B2H_D operator*(T a, const B2H_D& b) { return b * a; }
B2H_TN B2H_D operator/(const B2H_D& a, T b) { return a * ((T)1 / b); }
B2H_TN B2H_D operator/(T a, const B2H_D& b) { return B2H_D(a) / b; }
B2H_TN B2H_D& operator+=(B2H_D& a, const B2H_D& b) { a = a + b; return a; }
B2H_TN B2H_D& operator-=(B2H_D& a, const B2H_D& b) { a = a - b; return a; }
B2H_TN B2H_D& operator+=(B2H_D& a, T b) { a.v += b; return a; }
B2H_TN B2H_D& operator-=(B2H_D& a, T b) { a.v -= b; return a; }
B2H_TN B2H_D chain1(const B2H_D& a, T f, T df) { return b2h_node(f, a.id, df, -1, (T)0); }
)";

const char* kVarWrapper = R"(
__device__ inline void b2h_tape_begin(const B2hTape& t) {
    if (threadIdx.x == 0) b2h_tape = t;
    b2h_tape_count[threadIdx.x] = 0;
    __syncthreads();
}
// every thread of the block calls this (chains past C with count 0): one atomic per warp
__device__ inline void b2h_tape_end() {
    const int n = __reduce_max_sync(0xffffffffu, (unsigned)b2h_tape_count[threadIdx.x]);
    if ((threadIdx.x & 31) == 0 && n > 0) atomicMax((unsigned long long*)b2h_tape.needed, (unsigned long long)n);
}
template <typename T>
__device__ T potential_and_grad(const T* q, T* g, int d, const T* data) {
    typedef Var<T> S;
    const long long c = b2h_chain(), P = b2h_tape.pitch;
    T* adj = (T*)b2h_tape.adj;
    S x[B2H_AD_DIM];
    for (int i = 0; i < B2H_AD_DIM; ++i) { x[i].v = q[i]; x[i].id = i; adj[i * P + c] = (T)0; }
    const S lp = log_density<S, T>(x, B2H_AD_DIM, data);
    const int n = b2h_tape_count[threadIdx.x];
    if (n > b2h_tape.cap) {
        for (int i = 0; i < B2H_AD_DIM; ++i) g[i] = (T)0;
        return (T)__longlong_as_double(0x7ff0000000000000LL);    // +inf
    }
    if (lp.id >= 0) adj[lp.id * P + c] = (T)1;
    const T* pa0 = (const T*)b2h_tape.pa0;
    const T* pa1 = (const T*)b2h_tape.pa1;
    for (int k = n - 1; k >= 0; --k) {
        const long long e = (long long)k * P + c;
        const T a = adj[(long long)(B2H_AD_DIM + k) * P + c];
        const int i0 = b2h_tape.id0[e];
        if (i0 >= 0) adj[i0 * P + c] += pa0[e] * a;
        const int i1 = b2h_tape.id1[e];       // read after the first update: x * x adds both contributions
        if (i1 >= 0) adj[i1 * P + c] += pa1[e] * a;
    }
    for (int i = 0; i < B2H_AD_DIM; ++i) g[i] = -adj[i * P + c];
    return -lp.v;
}
)";

// The thread-per-chain kernels of every mode.  Only reverse mode uses the tape argument; the other modes get
// no-op hooks.
const char* kWrapper = R"(
#ifndef B2H_REVERSE
struct B2hTape { void* unused; };
__device__ inline void b2h_tape_begin(const B2hTape&) {}
__device__ inline void b2h_tape_end() {}
#endif
extern "C" __global__ void b2h_user_kernel_f64(const double* q, double* U, double* g, long long C, int d, const double* data, B2hTape tape) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    b2h_tape_begin(tape);
    if (c < C) U[c] = potential_and_grad<double>(q + c * d, g + c * d, d, data);
    b2h_tape_end();
}
extern "C" __global__ void b2h_user_kernel_f32(const float* q, float* U, float* g, long long C, int d, const float* data, B2hTape tape) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    b2h_tape_begin(tape);
    if (c < C) U[c] = potential_and_grad<float>(q + c * d, g + c * d, d, data);
    b2h_tape_end();
}
)";

}  // namespace

// host mirror of B2hTape in kVarHeader
struct TapeArgs {
    int* id0; int* id1; void* pa0; void* pa1; void* adj;
    long long pitch;
    int cap;
    long long* needed;
};

static i64 round256(i64 n) { return (n + 255) & ~(i64)255; }

// the reverse-mode tape layout of kVarHeader; returns the bytes the workspace needs
static i64 tape_layout(const b2h_user_model* um, int dtype, i64 C, char* ws, TapeArgs* t) {
    const i64 pitch = (C + 31) / 32 * 32, cap = um->tape_nodes, es = dtype == B2H_F64 ? 8 : 4;
    const i64 ids = round256(cap * pitch * 4), pas = round256(cap * pitch * es);
    const i64 adj = round256(((i64)um->dim + cap) * pitch * es);
    if (t) {
        char* b = (char*)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
        t->id0 = (int*)b; t->id1 = (int*)(b + ids);
        t->pa0 = b + 2 * ids; t->pa1 = b + 2 * ids + pas; t->adj = b + 2 * ids + 2 * pas;
        t->pitch = pitch; t->cap = (int)cap; t->needed = um->needed;
    }
    return 256 + 2 * ids + 2 * pas + adj;
}

i64 user_workspace_bytes(const b2h_model* m, int dtype, i64 C) {
    const b2h_user_model* um = (const b2h_user_model*)m->a;
    if (!um || !um->reverse || C <= 0) return 0;
    return tape_layout(um, dtype, C, nullptr, nullptr);
}

template <typename T>
int user_potential_and_grad(b2h_ctx* ctx, const b2h_model* m, const T* q, T* U, T* g, i64 C, void* ws, i64 ws_bytes) {
    const b2h_user_model* um = (const b2h_user_model*)m->a;
    if (!um) { set_error("user model: null handle (b2h_model.a must hold the b2h_user_model*)"); return B2H_ERR_ARG; }
    TapeArgs tape;
    memset(&tape, 0, sizeof(tape));
    if (um->reverse) {
        if (m->dim != um->dim) { set_error("user model: b2h_model.dim differs from the dim the handle was compiled for"); return B2H_ERR_ARG; }
        if (ctx->device != um->device) {
            set_error("user model: reverse-mode handle was created on device " + std::to_string(um->device) +
                      ", the context is on device " + std::to_string(ctx->device));
            return B2H_ERR_ARG;
        }
        const i64 need = tape_layout(um, Num<T>::dtype, C, (char*)ws, &tape);
        if (!ws || ws_bytes < need) {
            set_error("user model: workspace too small for the tape: need " + std::to_string(need) + " bytes");
            return B2H_ERR_WORKSPACE;
        }
    }
    long long Cl = C;
    int d = m->dim;
    const void* data = m->b;
    void* args[] = {(void*)&q, (void*)&U, (void*)&g, (void*)&Cl, (void*)&d, (void*)&data, (void*)&tape};
    const int threads = 128;     // B2H_TAPE_THREADS
    const unsigned grid = (unsigned)((C + threads - 1) / threads);
    B2H_CUDA(cudaLaunchKernel((const void*)(sizeof(T) == 8 ? um->k64 : um->k32), dim3(grid), dim3(threads), args, 0,
                              ctx->stream));
    return 0;
}
template int user_potential_and_grad<float>(b2h_ctx*, const b2h_model*, const float*, float*, float*, i64, void*, i64);
template int user_potential_and_grad<double>(b2h_ctx*, const b2h_model*, const double*, double*, double*, i64, void*,
                                             i64);

}  // namespace b2h

static int user_model_compile(const std::string& src, int ad_dim, bool reverse, b2h_user_model** out) {
    using namespace b2h;
    Nvrtc& rt = nvrtc();
    if (!rt.ok) { set_error("b2h_user_model_create: libnvrtc.so.12 not found (NVRTC is needed for user models)"); return B2H_ERR_UNSUPPORTED; }
    nvrtcProgram prog = nullptr;
    if (rt.CreateProgram(&prog, src.c_str(), "b2h_user_model.cu", 0, nullptr, nullptr) != 0) {
        set_error("nvrtcCreateProgram failed");
        return B2H_ERR_CUDA;
    }
    const std::string ad = "-DB2H_AD_DIM=" + std::to_string(ad_dim > 0 ? ad_dim : 1);
    const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "--fmad=false", ad.c_str()};
    const int rc = rt.CompileProgram(prog, 4, opts);
    if (rc != 0) {
        size_t n = 0;
        rt.GetProgramLogSize(prog, &n);
        std::string log(n, '\0');
        if (n) rt.GetProgramLog(prog, &log[0]);
        rt.DestroyProgram(&prog);
        set_error("user model does not compile:\n" + log);
        return B2H_ERR_ARG;
    }
    size_t nb = 0;
    rt.GetCUBINSize(prog, &nb);
    std::vector<char> cubin(nb);
    rt.GetCUBIN(prog, cubin.data());
    rt.DestroyProgram(&prog);
    b2h_user_model* um = new b2h_user_model();
    um->reverse = reverse;
    um->dim = ad_dim;
    cudaError_t e = cudaLibraryLoadData(&um->lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e == cudaSuccess) e = cudaLibraryGetKernel(&um->k64, um->lib, "b2h_user_kernel_f64");
    if (e == cudaSuccess) e = cudaLibraryGetKernel(&um->k32, um->lib, "b2h_user_kernel_f32");
    if (e == cudaSuccess && reverse) e = cudaGetDevice(&um->device);
    if (e == cudaSuccess && reverse) e = cudaMalloc((void**)&um->needed, sizeof(long long));
    if (e == cudaSuccess && reverse) e = cudaMemset(um->needed, 0, sizeof(long long));
    if (e != cudaSuccess) {
        set_error(std::string("user model: loading the compiled code failed: ") + cudaGetErrorString(e));
        if (um->needed) cudaFree(um->needed);
        delete um;
        return B2H_ERR_CUDA;
    }
    *out = um;
    return 0;
}

extern "C" int b2h_user_model_create(const char* cuda_source, b2h_user_model** out) {
    if (!cuda_source || !out) { b2h::set_error("b2h_user_model_create: null argument"); return B2H_ERR_ARG; }
    return user_model_compile(std::string(cuda_source) + b2h::kWrapper, 0, false, out);
}

extern "C" int b2h_user_model_create_ad(const char* cuda_source, int32_t dim, b2h_user_model** out) {
    if (!cuda_source || !out) { b2h::set_error("b2h_user_model_create_ad: null argument"); return B2H_ERR_ARG; }
    if (dim < 1 || dim > 64) { b2h::set_error("b2h_user_model_create_ad: dim must be in [1, 64] (forward mode costs O(dim) per operation)"); return B2H_ERR_ARG; }
    return user_model_compile(std::string(b2h::kDualHeader) + b2h::kUnary + cuda_source + b2h::kDualWrapper +
                              b2h::kWrapper, dim, false, out);
}

extern "C" int b2h_user_model_create_rev(const char* cuda_source, int32_t dim, b2h_user_model** out) {
    if (!cuda_source || !out) { b2h::set_error("b2h_user_model_create_rev: null argument"); return B2H_ERR_ARG; }
    if (dim < 1 || dim > B2H_USER_REV_MAX_DIM) {
        b2h::set_error("b2h_user_model_create_rev: dim must be in [1, " + std::to_string(B2H_USER_REV_MAX_DIM) + "]");
        return B2H_ERR_ARG;
    }
    return user_model_compile(std::string(b2h::kVarHeader) + b2h::kUnary + cuda_source + b2h::kVarWrapper +
                              b2h::kWrapper, dim, true, out);
}

extern "C" int b2h_user_model_set_tape_nodes(b2h_user_model* um, int64_t nodes) {
    if (!um || !um->reverse) { b2h::set_error("b2h_user_model_set_tape_nodes: needs a reverse-mode handle"); return B2H_ERR_ARG; }
    if (nodes < 0 || nodes > (int64_t)INT32_MAX - um->dim) {
        b2h::set_error("b2h_user_model_set_tape_nodes: nodes must be in [0, 2^31 - 1 - dim]");
        return B2H_ERR_ARG;
    }
    um->tape_nodes = nodes;
    return 0;
}

extern "C" int b2h_user_model_tape_needed(b2h_ctx* ctx, b2h_user_model* um, int64_t* needed) {
    if (!ctx || !um || !needed || !um->reverse) { b2h::set_error("b2h_user_model_tape_needed: bad argument (needs a reverse-mode handle)"); return B2H_ERR_ARG; }
    if (ctx->device != um->device) { b2h::set_error("b2h_user_model_tape_needed: the context is on another device than the handle"); return B2H_ERR_ARG; }
    long long h = 0;
    B2H_CUDA(cudaMemcpyAsync(&h, um->needed, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    B2H_CUDA(cudaMemsetAsync(um->needed, 0, sizeof(long long), ctx->stream));
    B2H_CUDA(cudaStreamSynchronize(ctx->stream));
    *needed = h;
    return 0;
}

extern "C" int b2h_user_model_destroy(b2h_user_model* um) {
    if (!um) return 0;
    cudaLibraryUnload(um->lib);
    if (um->needed) cudaFree(um->needed);
    delete um;
    return 0;
}
