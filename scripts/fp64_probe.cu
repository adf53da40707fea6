// FP64 FMA rate probe for scripts/fir_f64_time.py: every thread runs 8 independent DFMA chains, so the FP64 pipe,
// not the FMA latency, bounds the kernel.  Built by the script with nvcc -shared (sm_100a) and called through ctypes.
#include <cuda_runtime.h>

constexpr int CHAINS = 8;

__global__ void __launch_bounds__(256) fp64_probe_kernel(double *out, int iters, double a, double b)
{
    double acc[CHAINS];
#pragma unroll
    for (int i = 0; i < CHAINS; ++i) acc[i] = threadIdx.x * 1e-3 + i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < CHAINS; ++i) acc[i] = fma(acc[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < CHAINS; ++i) s += acc[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// DFMA executed by one launch: blocks * 256 * iters * CHAINS
extern "C" int fp64_probe_launch(double *out, int blocks, int iters, double a, double b, void *stream)
{
    fp64_probe_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(out, iters, a, b);
    return (int)cudaGetLastError();
}

extern "C" int fp64_probe_chains() { return CHAINS; }
