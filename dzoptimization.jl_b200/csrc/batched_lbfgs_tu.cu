// batched_lbfgs_tu.cu -- instantiates the batched live L-BFGS kernel for every even n <= DZO_SMALL_N_MAX in its own
// translation unit (dzopt_lbfgs.cu launches it through these pointers; keeps the sixteen ptxas jobs in parallel with the
// others).
#include "batched_lbfgs.cuh"

namespace dzo {

const void* batched_lbfgs_kernel_ptr(int n) {
    switch (n) {
        case 2: return (const void*)batched_lbfgs_kernel<2>;
        case 4: return (const void*)batched_lbfgs_kernel<4>;
        case 6: return (const void*)batched_lbfgs_kernel<6>;
        case 8: return (const void*)batched_lbfgs_kernel<8>;
        case 10: return (const void*)batched_lbfgs_kernel<10>;
        case 12: return (const void*)batched_lbfgs_kernel<12>;
        case 14: return (const void*)batched_lbfgs_kernel<14>;
        case 16: return (const void*)batched_lbfgs_kernel<16>;
        case 18: return (const void*)batched_lbfgs_kernel<18>;
        case 20: return (const void*)batched_lbfgs_kernel<20>;
        case 22: return (const void*)batched_lbfgs_kernel<22>;
        case 24: return (const void*)batched_lbfgs_kernel<24>;
        case 26: return (const void*)batched_lbfgs_kernel<26>;
        case 28: return (const void*)batched_lbfgs_kernel<28>;
        case 30: return (const void*)batched_lbfgs_kernel<30>;
        case 32: return (const void*)batched_lbfgs_kernel<32>;
        default: return nullptr;
    }
}

// public column-major n x batch (problem p at p*n + e) <-> the kernel's batch-innermost layout (e*batch + p)
static __global__ void batched_lbfgs_transpose_kernel(const double* __restrict__ src, double* __restrict__ dst, int n,
                                                      long long batch, int to_public) {
    const long long total = (long long)n * batch;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i / n, e = i - p * n;
        if (to_public) dst[i] = src[e * batch + p];
        else dst[e * batch + p] = src[i];
    }
}

cudaError_t batched_lbfgs_transpose(const double* src, double* dst, int n, long long batch, int to_public,
                                    cudaStream_t stream) {
    const long long total = (long long)n * batch;
    const long long blocks = (total + 255) / 256;
    batched_lbfgs_transpose_kernel<<<(unsigned)(blocks < 65536 ? blocks : 65536), 256, 0, stream>>>(src, dst, n, batch,
                                                                                                     to_public);
    return cudaGetLastError();
}

}  // namespace dzo
