// NcoNode batching shim (SURVEY 8(f) rank 4): Nco::push (src/demodulation/nco.rs:71-77) over a batch of phase errors.
//
// The reference is a one-sample recurrence  phase += dphase + perr; if phase > 2 pi { phase -= 2 pi };  out = e^{j phase}.
// Over a batch the phase after sample k is (mod 2 pi)
//     phase0 + (k+1) * dphase + sum_{i<=k} perr[i],
// i.e. an inclusive prefix sum of perr plus an arithmetic ramp -- a scan, not a recurrence.  The ramp term is formed
// exactly ((k+1)*dphase as an FMA two-product) and reduced against a four-part 2 pi, so it does not accumulate
// rounding the way n sequential additions do; the prefix sum runs over perr alone (small numbers in a loop filter), in
// f64, block-wise.  The single conditional wrap of the reference only changes the representative of the phase mod 2 pi,
// never e^{j phase}.
//
// Three launches per call: (1) per-tile sums of perr, (2) exclusive scan of the tile sums (one CTA), (3) per-tile scan +
// phase + sincos.  HBM: perr is read twice (8 + 8 B), the output written once (16 B): 24 B per sample algorithmic at
// 8 B in + 16 B out; FP64-bound in practice (sincos in f64).
#include "common.cuh"
#include "misc_kernels.cuh"

namespace cb {

constexpr int NCO_THREADS = 256;
constexpr int NCO_PER_THREAD = 8;
constexpr int NCO_TILE = NCO_THREADS * NCO_PER_THREAD;

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(NCO_THREADS) nco_tile_sum_kernel(const double *__restrict__ perr, size_t n, double *__restrict__ tile_sum)
{
    __shared__ double ws[NCO_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * NCO_TILE + (size_t)threadIdx.x * NCO_PER_THREAD;
    double s = 0.0;
    if (base + NCO_PER_THREAD <= n && (reinterpret_cast<uintptr_t>(perr) & 15) == 0) {
        const double2 *p = reinterpret_cast<const double2 *>(perr + base);
#pragma unroll
        for (int i = 0; i < NCO_PER_THREAD / 2; ++i) {
            const double2 v = __ldg(p + i);
            s += v.x;
            s += v.y;
        }
    } else {
        for (int i = 0; i < NCO_PER_THREAD; ++i)
            if (base + i < n) s += perr[base + i];
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < NCO_THREADS / 32; ++w) t += ws[w];
        tile_sum[blockIdx.x] = t;
    }
}

// r = x mod 2 pi in [-pi, pi] for x = k * d given as the exact pair (hi, lo) with k*d = hi + lo; q * C1..C3 are exact
// for q < 2^29 (24-bit pieces of 2 pi)
__device__ __forceinline__ double reduce_2pi(double hi, double lo)
{
    const double inv2pi = 0.15915494309189534561;
    const double C1 = 0x1.921fb40000000p+2, C2 = 0x1.4442d00000000p-22, C3 = 0x1.8469880000000p-46,
                 C4 = 0x1.8cc51701b839ap-70;
    const double q = rint(hi * inv2pi);
    double r = fma(-q, C1, hi);
    r = fma(-q, C2, r);
    r = fma(-q, C3, r);
    r = fma(-q, C4, r);
    return r + lo;
}

// exclusive scan of the tile sums in place, one CTA of 1024 threads, chunks of 1024 with a running carry; prefixes are
// stored reduced mod 2 pi so that their magnitude (and rounding) does not grow with the batch length
__global__ void __launch_bounds__(1024) nco_scan_tiles_kernel(double *__restrict__ tile_sum, size_t ntiles)
{
    __shared__ double ws[32];
    __shared__ double carry_s;
    if (threadIdx.x == 0) carry_s = 0.0;
    __syncthreads();
    for (size_t c = 0; c < ntiles; c += 1024) {
        const size_t i = c + threadIdx.x;
        const double v = i < ntiles ? tile_sum[i] : 0.0;
        double incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        // exclusive prefix by shifting the inclusive scan up one lane, never as incl - v: a non-finite or huge tile sum
        // must not reach the prefixes of the tiles before it
        double excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if ((threadIdx.x & 31) == 0) excl = 0.0;
        if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            double w = ws[threadIdx.x];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, w, o);
                if (threadIdx.x >= o) w += t;
            }
            ws[threadIdx.x] = w;
        }
        __syncthreads();
        const double before_warp = (threadIdx.x >> 5) ? ws[(threadIdx.x >> 5) - 1] : 0.0;
        const double carry = carry_s;
        if (i < ntiles) tile_sum[i] = reduce_2pi(carry + before_warp + excl, 0.0);
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = reduce_2pi(carry + before_warp + incl, 0.0);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(NCO_THREADS) nco_apply_kernel(const double *__restrict__ perr, size_t n, const double *__restrict__ tile_pre,
                                                                const double *__restrict__ phase_in, double *__restrict__ phase_out,
                                                                double dphase, double2 *__restrict__ out)
{
    __shared__ double ws[NCO_THREADS / 32];
    const size_t base = (size_t)blockIdx.x * NCO_TILE + (size_t)threadIdx.x * NCO_PER_THREAD;
    double v[NCO_PER_THREAD];
    if (base + NCO_PER_THREAD <= n && (reinterpret_cast<uintptr_t>(perr) & 15) == 0) {
        const double2 *p = reinterpret_cast<const double2 *>(perr + base);
#pragma unroll
        for (int i = 0; i < NCO_PER_THREAD / 2; ++i) {
            const double2 t = __ldg(p + i);
            v[2 * i] = t.x;
            v[2 * i + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < NCO_PER_THREAD; ++i) v[i] = base + i < n ? perr[base + i] : 0.0;
    }
#pragma unroll
    for (int i = 1; i < NCO_PER_THREAD; ++i) v[i] += v[i - 1];  // thread-local inclusive scan
    double incl = v[NCO_PER_THREAD - 1];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incl, o);
        if ((threadIdx.x & 31) >= o) incl += t;
    }
    // exclusive prefix of the lanes before this one (shifted scan, not incl - mine: output k depends on perr[0..k] only,
    // so a NaN, an Inf or one huge value cannot change or cancel into the outputs before it)
    double excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if ((threadIdx.x & 31) == 0) excl = 0.0;
    if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    double off = tile_pre[blockIdx.x] + excl;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) off += ws[w];
    const double ph0 = *phase_in;
#pragma unroll
    for (int i = 0; i < NCO_PER_THREAD; ++i) {
        const size_t k = base + i;
        if (k < n) {
            const double kd = (double)(k + 1);
            const double hi = kd * dphase;
            const double lo = fma(kd, dphase, -hi);
            const double ph = ph0 + reduce_2pi(hi, lo) + (off + v[i]);
            double sn, cs;
            sincos(ph, &sn, &cs);
            out[k] = make_double2(cs, sn);
            if (k == n - 1) {  // carried phase, kept in [0, 2 pi)
                double r = reduce_2pi(ph, 0.0);
                if (r < 0.0) r += 6.283185307179586476925;
                *phase_out = r;
            }
        }
    }
}

size_t nco_scratch_doubles(size_t n) { return ceil_div(n, (size_t)NCO_TILE); }

int launch_nco(const double *perr, size_t n, double *tile_scratch, const double *phase_in, double *phase_out, double dphase,
               double2 *out, cudaStream_t s)
{
    CB_REQUIRE(n < ((size_t)1 << 29), CB_ERR_UNSUPPORTED, "nco: at most 2^29 - 1 phase errors per call");
    const size_t ntiles = ceil_div(n, (size_t)NCO_TILE);
    nco_tile_sum_kernel<<<(unsigned)ntiles, NCO_THREADS, 0, s>>>(perr, n, tile_scratch);
    count_launch();
    nco_scan_tiles_kernel<<<1, 1024, 0, s>>>(tile_scratch, ntiles);
    count_launch();
    nco_apply_kernel<<<(unsigned)ntiles, NCO_THREADS, 0, s>>>(perr, n, tile_scratch, phase_in, phase_out, dphase, out);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

}  // namespace cb
