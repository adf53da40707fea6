// Complex<f64> FFT kernels for sm_100a (cb_fft_f64).  Every rounding happens in the host/device functions of
// fft64_core.cuh; this file only maps butterflies to threads and points to memory.
#include "fft64_core.cuh"
#include "fft_f64_kernels.cuh"

namespace cb {

using namespace f64fft;

namespace {

constexpr int MAX_THREADS = 512;  // CTA_POINTS / 8 columns, or one 4096-point frame, or 4 columns of 1024 points

__device__ __forceinline__ z64 ldg(const z64 *p)
{
    const double2 v = __ldg(reinterpret_cast<const double2 *>(p));
    return {v.x, v.y};
}

// shared-memory slot of point e of a column: one pad slot per 8 points, so that the first pass's stores (8 points
// apart per thread) hit 8 distinct 16-byte banks per quarter warp; the column pitch is odd for the same reason when
// consecutive threads hold consecutive columns
__device__ __forceinline__ unsigned spad(unsigned e) { return e + (e >> 3); }

// One radix-R Stockham pass at stride p over the CTA's columns; each thread does 8 / R butterflies.  The first pass
// reads global memory, the last one writes it; the others work in place in shared memory (all reads, a barrier, all
// writes).  Consecutive threads take consecutive columns where the global side is contiguous over columns (c_fast),
// else consecutive butterflies of one column.
template <int R, bool INV>
__device__ __forceinline__ void cols_pass(const Fft64Cols &a, z64 *sm, unsigned pitch, size_t f, unsigned c0,
                                          unsigned B, unsigned p, bool first, bool last)
{
    constexpr int PER = 8 / R;
    const unsigned n = 1u << a.log2n, nb = n / R;
    const bool c_fast = first ? a.in_c == 1 : (last ? a.out_c == 1 : false);
    const z64 *in = reinterpret_cast<const z64 *>(a.in);
    z64 *out = reinterpret_cast<z64 *>(a.out);
    z64 v[8];
    unsigned cs[PER], is[PER];
#pragma unroll
    for (int r = 0; r < PER; ++r) {
        const unsigned b = threadIdx.x + r * blockDim.x;
        const unsigned c = c_fast ? b % B : b / nb, i = c_fast ? b / B : b % nb;
        cs[r] = c;
        is[r] = i;
        const unsigned col = c0 + c;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const unsigned e = i + j * nb;
            if (first)
                v[r * R + j] = col < a.cols ? ldg(in + f * a.in_f + col * a.in_c + e * a.in_j) : z64{0.0, 0.0};
            else
                v[r * R + j] = sm[c * pitch + spad(e)];
        }
    }
    if (!first) __syncthreads();  // every read of the pass before any in-place write
#pragma unroll
    for (int r = 0; r < PER; ++r) {
        const unsigned c = cs[r], i = is[r], k = i & (p - 1), col = c0 + c;
        stockham_bfly<R, INV>(v + r * R, reinterpret_cast<const z64 *>(a.tw), k, a.tw_step * (n / (p * R)));
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const unsigned e = (i - k) * R + k + j * p;
            if (last) {
                if (col < a.cols) {
                    z64 y = v[r * R + j];
                    const size_t t = (size_t)e * col;
                    if (a.twist && t) y = cmul(y, ldg(reinterpret_cast<const z64 *>(a.twist) + t));
                    reinterpret_cast<double2 *>(out + f * a.out_f + col * a.out_c + e * a.out_k)[0] = make_double2(y.re, y.im);
                }
            } else {
                sm[c * pitch + spad(e)] = v[r * R + j];
            }
        }
    }
    if (!last) __syncthreads();
}

// One CTA = B columns (sub-transforms) of one frame: radix-8 passes, then one radix-4 or radix-2 pass when log2n is
// not a multiple of 3.
template <bool INV>
__global__ void __launch_bounds__(MAX_THREADS) fft64_cols_kernel(const __grid_constant__ Fft64Cols a, unsigned B,
                                                                 unsigned blocks_per_frame)
{
    extern __shared__ __align__(16) unsigned char fsm[];
    z64 *sm = reinterpret_cast<z64 *>(fsm);
    const unsigned L = a.log2n, pitch = spad(1u << L) | 1u;
    const size_t f = blockIdx.x / blocks_per_frame;
    const unsigned c0 = (blockIdx.x % blocks_per_frame) * B;
    const unsigned n8 = L / 3, rem = L % 3, np = n8 + (rem ? 1 : 0);
    unsigned p = 1;
    for (unsigned ps = 0; ps < n8; ++ps, p *= 8) cols_pass<8, INV>(a, sm, pitch, f, c0, B, p, ps == 0, ps + 1 == np);
    if (rem == 2) cols_pass<4, INV>(a, sm, pitch, f, c0, B, p, false, true);
    if (rem == 1) cols_pass<2, INV>(a, sm, pitch, f, c0, B, p, false, true);
}

// one thread per output bin: X[k] = sum_n x[n] tw[kn mod N] in ascending n, the index advanced exactly
__global__ void __launch_bounds__(256) fft64_direct_kernel(const double2 *__restrict__ in, double2 *__restrict__ out,
                                                           const double2 *__restrict__ tw, unsigned N, size_t total)
{
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        const unsigned k = (unsigned)(g % N);
        const z64 *x = reinterpret_cast<const z64 *>(in) + (g - k);
        z64 acc{0.0, 0.0};
        unsigned e = 0;
        for (unsigned t = 0; t < N; ++t) {
            acc = direct_term(acc, ldg(x + t), ldg(reinterpret_cast<const z64 *>(tw) + e));
            e += k;
            if (e >= N) e -= N;
        }
        out[g] = make_double2(acc.re, acc.im);
    }
}

__global__ void __launch_bounds__(256) fft64_chirp_pre_kernel(const double2 *__restrict__ x, const double2 *__restrict__ chirp,
                                                              double2 *__restrict__ a, unsigned N, unsigned M, size_t total)
{
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        const size_t f = g / M;
        const unsigned t = (unsigned)(g - f * M);
        z64 y{0.0, 0.0};
        if (t < N) y = cmul(ldg(reinterpret_cast<const z64 *>(x) + f * N + t), ldg(reinterpret_cast<const z64 *>(chirp) + t));
        a[g] = make_double2(y.re, y.im);
    }
}

__global__ void __launch_bounds__(256) fft64_chirp_mul_kernel(double2 *__restrict__ spec, const double2 *__restrict__ bspec,
                                                              unsigned M, size_t total)
{
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        const double2 s = spec[g];
        const z64 y = cmul({s.x, s.y}, ldg(reinterpret_cast<const z64 *>(bspec) + g % M));
        spec[g] = make_double2(y.re, y.im);
    }
}

__global__ void __launch_bounds__(256) fft64_chirp_post_kernel(const double2 *__restrict__ c, const double2 *__restrict__ chirp,
                                                               double2 *__restrict__ out, unsigned N, unsigned M, size_t total)
{
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
        const size_t f = g / N;
        const unsigned k = (unsigned)(g - f * N);
        const z64 y = cmul(ldg(reinterpret_cast<const z64 *>(c) + f * M + k), ldg(reinterpret_cast<const z64 *>(chirp) + k));
        out[g] = make_double2(y.re, y.im);
    }
}

unsigned elem_grid(size_t total)
{
    const size_t g = ceil_div(total, (size_t)256);
    return (unsigned)(g < 148 * 32 ? g : 148 * 32);
}

}  // namespace

int launch_fft64_cols(const Fft64Cols &a, int inverse, cudaStream_t s)
{
    const bool col_major = a.in_c == 1;  // the columns of a two-step transform, not whole frames
    const unsigned B = cols_per_cta(a.log2n, col_major), n = 1u << a.log2n;
    const unsigned threads = B * n / 8, bpf = (unsigned)ceil_div(a.cols, B);
    const size_t smem = a.log2n > 3 ? (size_t)B * ((n + n / 8) | 1u) * sizeof(double2) : 0;
    const size_t grid = a.frames * bpf;
    if (grid == 0) return CB_OK;
    auto k = inverse ? fft64_cols_kernel<true> : fft64_cols_kernel<false>;
    CB_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<(unsigned)grid, threads, smem, s>>>(a, B, bpf);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

int launch_fft64_direct(const double2 *in, double2 *out, const double2 *tw, unsigned n, size_t frames, cudaStream_t s)
{
    const size_t total = frames * n;
    fft64_direct_kernel<<<elem_grid(total), 256, 0, s>>>(in, out, tw, n, total);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

int launch_fft64_chirp_pre(const double2 *x, const double2 *chirp, double2 *a, unsigned n, unsigned m, size_t frames,
                           cudaStream_t s)
{
    const size_t total = frames * m;
    fft64_chirp_pre_kernel<<<elem_grid(total), 256, 0, s>>>(x, chirp, a, n, m, total);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

int launch_fft64_chirp_mul(double2 *spec, const double2 *bspec, unsigned m, size_t frames, cudaStream_t s)
{
    const size_t total = frames * m;
    fft64_chirp_mul_kernel<<<elem_grid(total), 256, 0, s>>>(spec, bspec, m, total);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

int launch_fft64_chirp_post(const double2 *c, const double2 *chirp, double2 *out, unsigned n, unsigned m, size_t frames,
                            cudaStream_t s)
{
    const size_t total = frames * n;
    fft64_chirp_post_kernel<<<elem_grid(total), 256, 0, s>>>(c, chirp, out, n, m, total);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

}  // namespace cb
