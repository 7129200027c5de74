// Exhaustive check of the low residual piece of the fp16 x 2 fused logistic gradient: for every fp32 bit pattern rr,
// the piece as tc_gemm.cu forms it (rr + (-h) in one mixed f16 / f32 add, h = fp16(rr)) against the earlier form
// (h unpacked to f32, then an f32 add).  Prints the number of patterns whose fp16 bits differ, and how many have an
// fp16-exact rr (low piece +0: the sign-of-zero case).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o fused16_lo_piece benchmarks/micro/fused16_lo_piece.cu
#include <cstdio>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

__device__ __forceinline__ float sub_f16(float rr, __half h) {   // as in tc_gemm.cu
    float d;
    asm("{\n.reg .b16 n;\nneg.f16 n, %1;\nadd.rn.f32.f16 %0, n, %2;\n}" : "=f"(d) : "h"(__half_as_ushort(h)), "f"(rr));
    return d;
}

__global__ void check(unsigned long long* diff, unsigned long long* exact) {
    unsigned long long nd = 0, ne = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < (1ull << 32); i += stride) {
        const float rr = __uint_as_float((unsigned)i);
        const __half h = __float2half_rn(rr);
        float hf = __half2float(h);
        asm volatile("" : "+f"(hf));   // keep the old form's separate unpack and f32 add
        const __half lo_old = __float2half_rn(rr + (-hf));
        const __half lo_new = __float2half_rn(sub_f16(rr, h));
        nd += __half_as_ushort(lo_old) != __half_as_ushort(lo_new);
        ne += __half_as_ushort(lo_new) == 0;
    }
    atomicAdd(diff, nd);
    atomicAdd(exact, ne);
}

int main() {
    unsigned long long* c;
    if (cudaMallocManaged(&c, 2 * sizeof(unsigned long long)) != cudaSuccess) return 1;
    c[0] = c[1] = 0;
    check<<<148 * 8, 256>>>(c, c + 1);
    if (cudaDeviceSynchronize() != cudaSuccess) { printf("launch failed\n"); return 1; }
    printf("fp32 patterns: 4294967296, low piece bits differing: %llu, low piece +0: %llu\n", c[0], c[1]);
    const int rc = c[0] != 0;
    cudaFree(c);
    return rc;
}
