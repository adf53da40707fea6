// Complex<f64> FIR kernels for sm_100a (see fir_f64_kernels.cuh for the operation order they share).
//
// The hot path is the FP64 pipe: direct form with fused multiply-adds.  B200's data sheet gives the tensor path the
// same FP64 rate as the CUDA cores, so DMMA would buy nothing here.
#include "fir_f64_kernels.cuh"

namespace cb {

namespace {

constexpr int NT = 256;
constexpr int R = 8;            // consecutive outputs per thread
constexpr int TILE = NT * R;    // outputs per CTA step
constexpr int TK = 1024;        // taps per shared-memory chunk (a multiple of R)
constexpr unsigned MAX_CTAS = 148 * 4;  // stream kernel: grid-stride over tiles past MAX_CTAS * TILE outputs

// chain step of one output: the fixed order of the numerical contract (include/comms_b200.h)
template <bool CPLX>
__device__ __forceinline__ void fir64_term(double2 &acc, double2 h, double2 s)
{
    acc.x = fma(h.x, s.x, acc.x);
    if (CPLX) acc.x = fma(-h.y, s.y, acc.x);
    acc.y = fma(h.x, s.y, acc.y);
    if (CPLX) acc.y = fma(h.y, s.x, acc.y);
}

// sample idx of the stream [hist_in ++ x]: idx < 0 reads the history; anything the taps never reach reads as 0
__device__ __forceinline__ double2 fir64_sample(const Fir64Seg &a, long long idx)
{
    if (idx >= 0) return idx < (long long)a.n_in ? __ldg(a.x + idx) : make_double2(0.0, 0.0);
    const long long h = (long long)a.hist_len + idx;
    return h >= 0 ? __ldg(a.hist_in + h) : make_double2(0.0, 0.0);
}

__device__ __forceinline__ void fir64_write_hist(const Fir64Seg &a)
{
    const long long H = a.hist_len;
    for (long long i = threadIdx.x; i < H; i += blockDim.x) {
        const long long g = (long long)a.n_in - H + i;
        a.hist_out[i] = g >= 0 ? a.x[g] : a.hist_in[H + g];
    }
}

// ------------------------------------------------------------------------------------------------ stream kernel
// decim = interp = 1.  Thread t of a tile owns outputs t0 + R t + r, r < R.  For each chunk of up to TK taps the CTA
// stages the taps and the samples those taps reach for the tile in shared memory; the samples are stored
// de-interleaved by index mod R -- staged sample e at (e % R) * pitch + e / R, pitch odd -- so that the threads of a
// warp, whose windows are R samples apart, read consecutive 16-byte words, and the fill (consecutive e per thread)
// is conflict-free within each quarter warp.  Each thread slides an R-sample register window back over the stage: tap
// kk brings in one sample (one 16-byte load) and feeds R outputs (4 R or 2 R DFMA), the tap itself a broadcast load.
// The window slot of the sample at offset i (relative to the thread's first output) is i mod R, so with the tap loop
// unrolled by R every slot index is static.  A tap chunk's last group is guarded: padding taps never enter a chain.
template <bool CPLX>
__global__ void __launch_bounds__(NT, 2)
fir64_stream_kernel(const Fir64Seg a, const double2 *__restrict__ taps, unsigned pitch)
{
    extern __shared__ __align__(16) unsigned char fsm[];
    double2 *tsm = reinterpret_cast<double2 *>(fsm);  // complex taps of the chunk
    double *tsr = reinterpret_cast<double *>(fsm);    // real taps of the chunk
    double2 *xsm = reinterpret_cast<double2 *>(fsm + (size_t)TK * (CPLX ? sizeof(double2) : sizeof(double)));
    const int tid = threadIdx.x;
    const unsigned K = a.ntaps;
    if (a.hist_out != nullptr && blockIdx.x == 0) fir64_write_hist(a);
    const size_t ntiles = (a.n_in + TILE - 1) / TILE;
    for (size_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long t0 = (long long)tile * TILE;
        double2 acc[R];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = make_double2(0.0, 0.0);
        for (unsigned k0 = 0; k0 < K; k0 += TK) {
            const unsigned kc = K - k0 < (unsigned)TK ? K - k0 : (unsigned)TK;
            const unsigned kcr = (kc + R - 1) / R * R;
            __syncthreads();  // the previous chunk's (or tile's) reads are done
            for (unsigned i = tid; i < kc; i += NT) {
                const double2 h = __ldg(taps + k0 + i);
                if (CPLX) tsm[i] = h;
                else tsr[i] = h.x;
            }
            // staged e <-> sample t0 - k0 - (kcr - 1) + e, e < TILE + kcr - 1
            const long long s0 = t0 - (long long)k0 - (long long)(kcr - 1);
            for (unsigned e = tid; e < TILE + kcr - 1; e += NT) xsm[(e % R) * pitch + e / R] = fir64_sample(a, s0 + e);
            __syncthreads();
            // output r at tap kk reads staged e = R tid + kcr - 1 + r - kk: the sample at offset i = r - kk sits in
            // class (R - 1 + i) mod R, word tid + kcr / R - 1 + floor((R - 1 + i) / R)
            const double2 *wb = xsm + tid + kcr / R - 1;
            double2 w[R];
#pragma unroll
            for (int i = 1; i < R; ++i) w[i] = wb[(i - 1) * pitch + 1];
            const unsigned ng = kcr / R;
            for (unsigned g = 0; g < ng; ++g) {
                const bool full = (g + 1) * R <= kc;
#pragma unroll
                for (int jj = 0; jj < R; ++jj) {
                    const unsigned kk = g * R + jj;
                    if (full || kk < kc) {
                        w[(R - jj) % R] = wb[(R - 1 - jj) * pitch - g];  // offset -kk
                        const double2 h = CPLX ? tsm[kk] : make_double2(tsr[kk], 0.0);
#pragma unroll
                        for (int r = 0; r < R; ++r) fir64_term<CPLX>(acc[r], h, w[(r - jj + R) % R]);
                    }
                }
            }
        }
        // write back through shared memory (class r, word tid: conflict-free both ways) for coalesced stores
        __syncthreads();
        double2 *ysm = xsm;  // R * (NT + 1) <= R * pitch
#pragma unroll
        for (int r = 0; r < R; ++r) ysm[r * (NT + 1) + tid] = acc[r];
        __syncthreads();
        const long long rem = (long long)a.n_in - t0;
        const int nvalid = rem < TILE ? (int)rem : TILE;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const int o = j * NT + tid;
            if (o < nvalid) a.y[t0 + o] = ysm[(o % R) * (NT + 1) + o / R];
        }
    }
}

// ------------------------------------------------------------------------------------------------ resampling kernel
// decim D and / or interp L > 1: one surviving output per thread per step, only the non-zero-stuffed products.
//   q = output index, u = q D (zero-stuffed domain), p = u mod L, m = u / L:  y[q] = sum_j h[p + j L] * s[m - j]
template <bool CPLX>
__global__ void __launch_bounds__(256)
fir64_resample_kernel(const Fir64Seg a, const double2 *__restrict__ taps)
{
    if (a.hist_out != nullptr && blockIdx.x == 0) fir64_write_hist(a);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < a.n_out; q += stride) {
        const unsigned long long u = (unsigned long long)q * a.decim;
        const unsigned p = (unsigned)(u % a.interp);
        long long idx = (long long)(u / a.interp);
        double2 acc = make_double2(0.0, 0.0);
        for (unsigned k = p; k < a.ntaps; k += a.interp, --idx) {
            if ((long long)a.hist_len + idx < 0) break;  // older than the state: no term
            fir64_term<CPLX>(acc, __ldg(taps + k), fir64_sample(a, idx));
        }
        a.y[q] = acc;
    }
}

template <bool CPLX>
size_t stream_smem(unsigned pitch)
{
    return (size_t)TK * (CPLX ? sizeof(double2) : sizeof(double)) + (size_t)R * pitch * sizeof(double2);
}

template <bool CPLX>
int launch_stream64(const Fir64Seg &seg, const double2 *taps_dev, cudaStream_t s)
{
    const unsigned kmax = seg.ntaps < (unsigned)TK ? seg.ntaps : (unsigned)TK;
    const unsigned kcr = (kmax + R - 1) / R * R;
    const unsigned pitch = ((TILE + kcr) / R) | 1u;  // >= NT + 1 (the write-back layout) and odd
    const size_t smem = stream_smem<CPLX>(pitch);
    CB_CUDA(cudaFuncSetAttribute(fir64_stream_kernel<CPLX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    size_t grid = ceil_div(seg.n_in, (size_t)TILE);
    if (grid > MAX_CTAS) grid = MAX_CTAS;
    fir64_stream_kernel<CPLX><<<(unsigned)grid, NT, smem, s>>>(seg, taps_dev, pitch);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

template <bool CPLX>
int launch_resample64(const Fir64Seg &seg, const double2 *taps_dev, cudaStream_t s)
{
    size_t grid = ceil_div(seg.n_out ? seg.n_out : 1, (size_t)256);
    if (grid > 148 * 16) grid = 148 * 16;
    fir64_resample_kernel<CPLX><<<(unsigned)grid, 256, 0, s>>>(seg, taps_dev);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

}  // namespace

int launch_fir_f64(const Fir64Seg &seg, const double2 *taps_dev, bool taps_real, cudaStream_t stream)
{
    if (seg.n_in == 0) return CB_OK;
    if (seg.interp == 1 && seg.decim == 1)
        return taps_real ? launch_stream64<false>(seg, taps_dev, stream) : launch_stream64<true>(seg, taps_dev, stream);
    return taps_real ? launch_resample64<false>(seg, taps_dev, stream) : launch_resample64<true>(seg, taps_dev, stream);
}

}  // namespace cb
