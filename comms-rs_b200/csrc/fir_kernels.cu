// FIR kernels for sm_100a: overlap-save stream kernel (TMA-staged tiles with
// halo, taps in the kernel-parameter constant bank, packed FFMA2 inner loop)
// plus a generic any-shape kernel (interp / decim / long filters).
#include "chain_kernels.cuh"
#include "fir_kernels.cuh"

namespace cb {

// ============================================================================
// Stream kernel: decim = interp = 1, taps <= KP (zero padded), KP in {16,32,64,128}
//
// Tile = 256 threads x R consecutive outputs.  The input tile (TILE + KP samples,
// the first KP being the halo) lives in shared memory in chunks of R samples;
// each chunk is padded by 16 bytes so that the per-thread 128-bit window loads
// (lane stride = one chunk) are bank-conflict free.  Chunks are fetched with TMA
// 1-D bulk copies (UBLKCP) that complete on one mbarrier.
//
// Inner loop: for tap j (descending k), R accumulators += h * window -- one
// FFMA2 (two FP32 FMAs: re and im) per sample-tap for real-valued taps, two for
// complex taps (A += hr*(xr,xi); B += hi*(xr,xi); y = (A.x - B.y, A.y + B.x)).
// The tap operand comes from the constant bank (uniform register), so each
// FFMA2 reads two 64-bit vector registers only.
// Algorithmic HBM traffic: 8 B read + 8 B written per sample.
// ============================================================================

template <int KP, bool CPLX>
struct TapBank {
    // real: t[k] = (h[k], h[k]);  complex: t[2k] = (hr,hr), t[2k+1] = (hi,hi)
    float2 t[CPLX ? 2 * KP : KP];
};

struct StreamArgs {
    const float2 *x;
    const float2 *halo;  // KP samples preceding x[0]
    float2 *y;
    const float2 *hist_in;
    float2 *hist_out;
    unsigned long long n;
    unsigned hist_len;
    int aligned;  // x, y, halo 16-byte aligned -> TMA loads + 128-bit stores
};

template <int KP, bool CPLX, int R>
__global__ void __launch_bounds__(256, 2)
fir_stream_kernel(const __grid_constant__ StreamArgs a, const __grid_constant__ TapBank<KP, CPLX> taps)
{
    constexpr int NT = 256;
    constexpr int TILE = NT * R;
    constexpr int CHB = 8 * R;        // chunk bytes
    constexpr int STRIDE = CHB + 16;  // padded chunk pitch
    constexpr int NCH = (TILE + KP) / R;
    static_assert(KP % R == 0 && R % 2 == 0, "halo must be whole chunks");

    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;

    const int tid = threadIdx.x;
    const unsigned long long t0 = (unsigned long long)blockIdx.x * TILE;
    const unsigned long long rem = a.n - t0;
    const int nvalid = rem < (unsigned long long)TILE ? (int)rem : TILE;
    const int nbuf = KP + nvalid;  // valid samples in the tile buffer
    // buffer index i <-> sample x[t0 - KP + i]; for tile 0 the first KP come from a.halo
    const float2 *src_main = a.x + t0 - KP;  // only dereferenced for i >= KP when t0 == 0

    if (a.aligned) {
        if (tid == 0) {
            mbar_init(&bar, 1);
            fence_mbar_init();
        }
        __syncthreads();
        const int nfull = nbuf / R;
        const int tail = nbuf - nfull * R;          // samples in the partial chunk
        const int tail16 = (tail >> 1) << 1;        // whole 16-byte pairs of it
        if (tid < 32) {
            if (tid == 0) mbar_arrive_expect_tx(&bar, (uint32_t)(nfull * CHB + tail16 * 8));
            for (int c = tid; c < nfull; c += 32) {
                const float2 *src = (t0 == 0 && c < KP / R) ? a.halo + c * R : src_main + c * R;
                tma_load_1d(smem + c * STRIDE, src, CHB, &bar);
            }
            if (tid == 0 && tail16 > 0) tma_load_1d(smem + nfull * STRIDE, src_main + nfull * R, tail16 * 8, &bar);
        }
        if (tid == 32 && (tail & 1)) {  // odd last sample: plain copy
            *reinterpret_cast<float2 *>(smem + nfull * STRIDE + (tail - 1) * 8) = src_main[nfull * R + tail - 1];
        }
        mbar_wait(&bar, 0);
    } else {
        for (int i = tid; i < nbuf; i += NT) {
            const float2 v = (t0 == 0 && i < KP) ? a.halo[i] : src_main[i];
            *reinterpret_cast<float2 *>(smem + (i / R) * STRIDE + (i % R) * 8) = v;
        }
    }
    __syncthreads();

    // carried history for the next batch: last hist_len samples of [hist_in ++ x]
    if (a.hist_out != nullptr && blockIdx.x == gridDim.x - 1) {
        const long long H = a.hist_len;
        for (long long i = tid; i < H; i += NT) {
            const long long g = (long long)a.n - H + i;
            a.hist_out[i] = g >= 0 ? a.x[g] : a.hist_in[H + g];
        }
    }

    // ---- compute: thread tid owns outputs [R*tid, R*tid+R) of the tile.
    // output r needs buffer samples c = r + KP - k (k = tap index), relative to chunk `tid`.
    const unsigned char *base = smem + tid * STRIDE;
    constexpr int W = R + 2;  // rolling window, samples c in [j, j+R+1] live in wq[(c/2) % (W/2)]
    float4 wq[W / 2];
    auto ldpair = [&](int c) -> float4 {  // samples (c, c+1), c even
        return *reinterpret_cast<const float4 *>(base + (c / R) * STRIDE + (c % R) * 8);
    };
#pragma unroll
    for (int c = 0; c < W; c += 2) wq[(c / 2) % (W / 2)] = ldpair(c);

    float2 accA[R], accB[CPLX ? R : 1];
#pragma unroll
    for (int r = 0; r < R; ++r) accA[r] = make_float2(0.f, 0.f);
    if (CPLX) {
#pragma unroll
        for (int r = 0; r < (CPLX ? R : 1); ++r) accB[r] = make_float2(0.f, 0.f);
    }

    auto sample = [&](int c) -> float2 {
        const float4 q = wq[(c / 2) % (W / 2)];
        return (c & 1) ? make_float2(q.z, q.w) : make_float2(q.x, q.y);
    };

#pragma unroll
    for (int j = 0; j < KP; j += 2) {
        // taps k = KP-1-j and KP-2-j; sample for (r, k) is c = r + KP - k
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
            const int k = KP - 1 - j - jj;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const float2 s = sample(r + KP - k);
                if (CPLX) {
                    accA[r] = __ffma2_rn(s, taps.t[2 * k], accA[r]);
                    accB[r] = __ffma2_rn(s, taps.t[2 * k + 1], accB[r]);
                } else {
                    accA[r] = __ffma2_rn(s, taps.t[k], accA[r]);
                }
            }
        }
        // samples c = j, j+1 are dead now; bring in c = j+R+2, j+R+3
        if (j + 2 < KP) wq[((j + W) / 2) % (W / 2)] = ldpair(j + W);
    }

    // ---- store
    float2 *yo = a.y + t0 + (unsigned long long)tid * R;
    const int mine = nvalid - tid * R;  // outputs of this thread that exist
    if (mine >= R && a.aligned) {
#pragma unroll
        for (int r = 0; r < R; r += 2) {
            float4 v;
            if (CPLX) {
                v = make_float4(accA[r].x - accB[r].y, accA[r].y + accB[r].x, accA[r + 1].x - accB[r + 1].y,
                                accA[r + 1].y + accB[r + 1].x);
            } else {
                v = make_float4(accA[r].x, accA[r].y, accA[r + 1].x, accA[r + 1].y);
            }
            stg_stream(reinterpret_cast<float4 *>(yo + r), v);
        }
    } else {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (r < mine) {
                yo[r] = CPLX ? make_float2(accA[r].x - accB[r].y, accA[r].y + accB[r].x) : accA[r];
            }
        }
    }
}

// ============================================================================
// Generic kernel: any tap count, interp L, decim D.  One output per thread per
// step, taps and samples through L1.  Correct everywhere; used when no
// specialised kernel applies.
//   q = output index, u = q*D (zero-stuffed domain), p = u % L, m = u / L
//   y[q] = sum_j h[p + j*L] * s[m - j]
// ============================================================================
__global__ void __launch_bounds__(256)
fir_generic_kernel(FirSeg a, const float2 *__restrict__ taps)
{
    const long long H = a.hist_len;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < a.n_out; q += stride) {
        const unsigned long long u = (unsigned long long)q * a.decim;
        const unsigned p = (unsigned)(u % a.interp);
        const long long m = (long long)(u / a.interp);
        float ar = 0.f, ai = 0.f;
        long long idx = m;
        for (unsigned k = p; k < a.ntaps; k += a.interp, --idx) {
            float2 s;
            if (idx >= 0) s = a.x[idx];
            else if (H + idx >= 0) s = a.hist_in[H + idx];
            else break;  // older than any history: zeros
            const float2 h = __ldg(taps + k);
            ar = fmaf(h.x, s.x, ar);
            ar = fmaf(-h.y, s.y, ar);
            ai = fmaf(h.x, s.y, ai);
            ai = fmaf(h.y, s.x, ai);
        }
        a.y[q] = make_float2(ar, ai);
    }
    if (a.hist_out != nullptr && blockIdx.x == 0) {
        for (long long i = threadIdx.x; i < H; i += blockDim.x) {
            const long long g = (long long)a.n_in - H + i;
            a.hist_out[i] = g >= 0 ? a.x[g] : a.hist_in[H + g];
        }
    }
}

// ============================================================================
// Polyphase interpolator (K3): interp = L, taps-per-phase KPL (zero padded),
// decim = 1.  y[m*L + p] = sum_{j<KPL} h[p + j*L] * s[m - j].
// Same tiling as the stream kernel on the SYMBOL axis: thread owns R symbols
// and produces R*L outputs; never multiplies the stuffed zeros.
// Algorithmic HBM traffic: 8 B read + 8*L B written per symbol.
// ============================================================================
template <int L, int KPL>
struct PolyBank {
    float2 t[L * KPL];  // t[p*KPL + j] = (h[p+jL].re, h[p+jL].re): real taps only
};

template <int L, int KPL, int R>
__global__ void __launch_bounds__(256, 2)
fir_interp_kernel(const __grid_constant__ StreamArgs a, const __grid_constant__ PolyBank<L, KPL> taps)
{
    constexpr int NT = 256;
    constexpr int TILE = NT * R;  // symbols per tile
    constexpr int HALO = (KPL + R - 1) / R * R;
    constexpr int CHB = 8 * R;
    constexpr int STRIDE = CHB + 16;
    static_assert(R % 2 == 0, "R even");

    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar;

    const int tid = threadIdx.x;
    const unsigned long long t0 = (unsigned long long)blockIdx.x * TILE;
    const unsigned long long rem = a.n - t0;
    const int nvalid = rem < (unsigned long long)TILE ? (int)rem : TILE;
    const int nbuf = HALO + nvalid;
    const float2 *src_main = a.x + t0 - HALO;

    if (a.aligned) {
        if (tid == 0) {
            mbar_init(&bar, 1);
            fence_mbar_init();
        }
        __syncthreads();
        const int nfull = nbuf / R;
        const int tail = nbuf - nfull * R;
        const int tail16 = (tail >> 1) << 1;
        if (tid < 32) {
            if (tid == 0) mbar_arrive_expect_tx(&bar, (uint32_t)(nfull * CHB + tail16 * 8));
            for (int c = tid; c < nfull; c += 32) {
                const float2 *src = (t0 == 0 && c < HALO / R) ? a.halo + c * R : src_main + c * R;
                tma_load_1d(smem + c * STRIDE, src, CHB, &bar);
            }
            if (tid == 0 && tail16 > 0) tma_load_1d(smem + nfull * STRIDE, src_main + nfull * R, tail16 * 8, &bar);
        }
        if (tid == 32 && (tail & 1))
            *reinterpret_cast<float2 *>(smem + nfull * STRIDE + (tail - 1) * 8) = src_main[nfull * R + tail - 1];
        mbar_wait(&bar, 0);
    } else {
        for (int i = tid; i < nbuf; i += NT) {
            const float2 v = (t0 == 0 && i < HALO) ? a.halo[i] : src_main[i];
            *reinterpret_cast<float2 *>(smem + (i / R) * STRIDE + (i % R) * 8) = v;
        }
    }
    __syncthreads();

    if (a.hist_out != nullptr && blockIdx.x == gridDim.x - 1) {
        const long long H = a.hist_len;
        for (long long i = tid; i < H; i += NT) {
            const long long g = (long long)a.n - H + i;
            a.hist_out[i] = g >= 0 ? a.x[g] : a.hist_in[H + g];
        }
    }

    // symbol r of this thread is buffer index HALO + R*tid + r; tap j uses index - j
    const unsigned char *base = smem + tid * STRIDE;
    constexpr int NW = HALO + R;  // window samples c in [0, HALO+R) relative to chunk tid
    float2 w[NW];
#pragma unroll
    for (int c = 0; c < NW; c += 2) {
        const float4 q = *reinterpret_cast<const float4 *>(base + (c / R) * STRIDE + (c % R) * 8);
        w[c] = make_float2(q.x, q.y);
        w[c + 1] = make_float2(q.z, q.w);
    }
    float2 *yo = a.y + (t0 + (unsigned long long)tid * R) * L;
    const int mine = nvalid - tid * R;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        float2 acc[L];
#pragma unroll
        for (int p = 0; p < L; ++p) acc[p] = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = KPL - 1; j >= 0; --j) {
            const float2 s = w[HALO + r - j];
#pragma unroll
            for (int p = 0; p < L; ++p) acc[p] = __ffma2_rn(s, taps.t[p * KPL + j], acc[p]);
        }
        if (r < mine) {
            if (a.aligned && (L % 2 == 0)) {
#pragma unroll
                for (int p = 0; p < L; p += 2)
                    stg_stream(reinterpret_cast<float4 *>(yo + r * L + p),
                               make_float4(acc[p].x, acc[p].y, acc[p + 1].x, acc[p + 1].y));
            } else {
#pragma unroll
                for (int p = 0; p < L; ++p) yo[r * L + p] = acc[p];
            }
        }
    }
}

// ============================================================================
// launch wrappers
// ============================================================================
template <int KP, bool CPLX, int R>
static int launch_stream(const FirSeg &seg, const float2 *taps_host, cudaStream_t stream)
{
    TapBank<KP, CPLX> bank;
    for (int k = 0; k < KP; ++k) {
        const float2 h = k < (int)seg.ntaps ? taps_host[k] : make_float2(0.f, 0.f);
        if (CPLX) {
            bank.t[2 * k] = make_float2(h.x, h.x);
            bank.t[2 * k + 1] = make_float2(h.y, h.y);
        } else {
            bank.t[k] = make_float2(h.x, h.x);
        }
    }
    StreamArgs a;
    a.x = seg.x;
    a.halo = seg.hist_in + (seg.hist_len - KP);
    a.y = seg.y;
    a.hist_in = seg.hist_in;
    a.hist_out = seg.hist_out;
    a.n = seg.n_in;
    a.hist_len = seg.hist_len;
    a.aligned = ((reinterpret_cast<uintptr_t>(seg.x) | reinterpret_cast<uintptr_t>(seg.y) |
                  reinterpret_cast<uintptr_t>(a.halo)) & 15) == 0;
    constexpr int TILE = 256 * R;
    constexpr int SMEM = ((TILE + KP) / R) * (8 * R + 16);
    auto kern = fir_stream_kernel<KP, CPLX, R>;
        CB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    const unsigned grid = (unsigned)ceil_div(seg.n_in, (size_t)TILE);
    kern<<<grid, 256, SMEM, stream>>>(a, bank);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

template <int L, int KPL, int R>
static int launch_interp(const FirSeg &seg, const float2 *taps_host, cudaStream_t stream)
{
    PolyBank<L, KPL> bank;
    for (int p = 0; p < L; ++p)
        for (int j = 0; j < KPL; ++j) {
            const int k = p + j * L;
            const float h = k < (int)seg.ntaps ? taps_host[k].x : 0.f;
            bank.t[p * KPL + j] = make_float2(h, h);
        }
    constexpr int HALO = (KPL + R - 1) / R * R;
    StreamArgs a;
    a.x = seg.x;
    a.halo = seg.hist_in + (seg.hist_len - HALO);
    a.y = seg.y;
    a.hist_in = seg.hist_in;
    a.hist_out = seg.hist_out;
    a.n = seg.n_in;
    a.hist_len = seg.hist_len;
    a.aligned = ((reinterpret_cast<uintptr_t>(seg.x) | reinterpret_cast<uintptr_t>(seg.y) |
                  reinterpret_cast<uintptr_t>(a.halo)) & 15) == 0;
    constexpr int TILE = 256 * R;
    constexpr int SMEM = ((TILE + HALO) / R + 1) * (8 * R + 16);
    auto kern = fir_interp_kernel<L, KPL, R>;
        CB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    const unsigned grid = (unsigned)ceil_div(seg.n_in, (size_t)TILE);
    kern<<<grid, 256, SMEM, stream>>>(a, bank);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

static int launch_generic(const FirSeg &seg, const float2 *taps_dev, cudaStream_t stream)
{
    size_t blocks = ceil_div(seg.n_out ? seg.n_out : 1, (size_t)256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    fir_generic_kernel<<<(unsigned)blocks, 256, 0, stream>>>(seg, taps_dev);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

// Exact fall-back of the tensor-core filters: flagged tiles recomputed in f32 direct form, taps in order, and
// overwritten (see FirFix).  y[L m + p] = sum_q h[p + q L] * x[m - q]; x[-1-i] comes from the carried history.
__device__ __forceinline__ int fix_quant_i16(float v, float scale)  // Rust `(scale * v) as i16`: truncate, saturate, NaN -> 0
{
    const float t = v * scale;
    if (!(t == t)) return 0;
    return (int)fminf(fmaxf(truncf(t), -32768.f), 32767.f);
}

__global__ void __launch_bounds__(256) fir_fixup_kernel(const FirFixArgs a)
{
    const unsigned nfix = *a.count;
    const unsigned L = a.interp;
    for (unsigned t = blockIdx.x; t < nfix; t += gridDim.x) {
        const unsigned long long in0 = (unsigned long long)a.list[t] * a.tile_in;
        for (unsigned o = threadIdx.x; o < a.tile_in * L; o += blockDim.x) {
            const unsigned long long m = in0 + o / L;
            if (m >= a.n) break;
            const unsigned p = o % L;
            float re = 0.f, im = 0.f;
            long long idx = (long long)m;
            for (unsigned k = p; k < a.ntaps; k += L, --idx) {
                float2 xs = make_float2(0.f, 0.f);
                if (idx >= 0) {
                    if (a.x16 != nullptr) {
                        const uint32_t w = a.x16[idx];
                        xs = make_float2(__fmul_rn(a.in_scale, (float)(int16_t)(w & 0xFFFFu)), __fmul_rn(a.in_scale, (float)(int16_t)(w >> 16)));
                    } else {
                        xs = a.x[idx];
                    }
                }
                else if ((long long)a.hist_len + idx >= 0) xs = a.hist_in[(long long)a.hist_len + idx];
                const float2 h = __ldg(a.taps + k);
                re = fmaf(h.x, xs.x, re);
                re = fmaf(-h.y, xs.y, re);
                im = fmaf(h.x, xs.y, im);
                im = fmaf(h.y, xs.x, im);
            }
            const unsigned long long j = m * L + p;
            if (a.y16 != nullptr) {
                a.y16[2 * j] = (int16_t)fix_quant_i16(re, a.qscale);
                a.y16[2 * j + 1] = (int16_t)fix_quant_i16(im, a.qscale);
            } else {
                a.y[j] = make_float2(re, im);
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.next_count = 0;  // nobody else touches the other counter now
}

int launch_fir_fixup(const FirFixArgs &a, cudaStream_t stream)
{
    fir_fixup_kernel<<<148, 256, 0, stream>>>(a);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

bool fir_taps_pair_sparse(const float2 *taps, uint32_t ntaps, uint32_t interp)
{
    const uint32_t L = interp ? interp : 1;
    for (uint32_t p = 0; p < L; ++p) {
        bool any = false, even = false, odd = false;  // adjacent non-zero taps of this phase ending at an even / odd offset
        for (uint32_t q = 0; p + q * L < ntaps; ++q) {
            const float2 b = taps[p + q * L];
            if (b.x == 0.f && b.y == 0.f) continue;
            any = true;
            const float2 a = q ? taps[p + (q - 1) * L] : make_float2(0.f, 0.f);
            if (a.x != 0.f || a.y != 0.f) (q & 1 ? odd : even) = true;
        }
        if (any && !(even && odd)) return true;  // a phase without non-zero taps only ever outputs zeros
    }
    return false;
}

bool fir_fuses_i16(const FirSeg &seg, bool taps_real, const FirTcPlan *tcplan)
{
    return tcplan != nullptr && tcplan->bimg_dev != nullptr && seg.n_in >= tcplan->min_samples && seg.interp > 1 &&
           fir_ptc_applicable(seg, taps_real);
}

int launch_fir(const FirSeg &seg, const float2 *taps_dev, const float2 *taps_host, bool taps_real,
               const FirTcPlan *tcplan, cudaStream_t stream)
{
    if (seg.n_in == 0) return CB_OK;
    if (tcplan != nullptr && tcplan->bimg_dev != nullptr && seg.n_in >= tcplan->min_samples) {
        if (seg.interp == 1 && fir_tc_applicable(seg))
            return launch_fir_tc(seg, *tcplan, taps_dev, stream);
        if (seg.interp > 1 && fir_ptc_applicable(seg, taps_real)) return launch_fir_ptc(seg, *tcplan, taps_real, taps_dev, stream);
    }
    if (seg.interp == 1 && seg.decim == 1) {
        const uint32_t K = seg.ntaps;
        if (taps_real) {
            if (K <= 16 && seg.hist_len >= 16) return launch_stream<16, false, 16>(seg, taps_host, stream);
            if (K <= 32 && seg.hist_len >= 32) return launch_stream<32, false, 16>(seg, taps_host, stream);
            if (K <= 64 && seg.hist_len >= 64) return launch_stream<64, false, 16>(seg, taps_host, stream);
            if (K <= 128 && seg.hist_len >= 128) return launch_stream<128, false, 16>(seg, taps_host, stream);
        } else {
            if (K <= 16 && seg.hist_len >= 16) return launch_stream<16, true, 8>(seg, taps_host, stream);
            if (K <= 32 && seg.hist_len >= 32) return launch_stream<32, true, 8>(seg, taps_host, stream);
            if (K <= 64 && seg.hist_len >= 64) return launch_stream<64, true, 8>(seg, taps_host, stream);
            if (K <= 128 && seg.hist_len >= 128) return launch_stream<128, true, 8>(seg, taps_host, stream);
        }
    }
    // BatchFirNode -> DecimateNode with real taps: the fused bank kernel with one channel, no mixer and no FM tail
    // computes exactly this (only the surviving outputs, per-call decimation phase); TMA-staged for D in {5, 10}
    if (seg.interp == 1 && seg.decim > 1 && taps_real && seg.ntaps <= 64 && seg.n_in % 2 == 0 && seg.hist_len % 2 == 0 &&
        seg.hist_len >= 128 && (seg.decim == 2 || seg.decim == 4 || seg.decim == 5 || seg.decim == 8 || seg.decim == 10) &&
        (reinterpret_cast<uintptr_t>(seg.x) & 15) == 0 && (reinterpret_cast<uintptr_t>(seg.y) & 7) == 0) {
        ChainArgs a = {};
        a.x = seg.x;
        a.out = seg.y;
        a.hist_in = seg.hist_in;
        a.hist_out = seg.hist_out;  // may be NULL (host chunks before the last)
        a.n_in = seg.n_in;
        a.n_out = seg.n_out;
        a.ntaps = seg.ntaps;
        a.decim = seg.decim;
        a.hist_len = seg.hist_len;
        a.tile_out = 256;
        a.span_max = 256 * seg.decim + 64 + seg.decim;
        ChainTaps ct = {};
        for (uint32_t k = 0; k < seg.ntaps; ++k) ct.t[k] = make_float2(taps_host[k].x, taps_host[k].x);
        return launch_chain(a, ct, false, false, false, 1, stream);
    }
    if (seg.decim == 1 && taps_real && seg.interp > 1) {
        const uint32_t kpl = (uint32_t)ceil_div(seg.ntaps, seg.interp);
        if (seg.interp == 4 && kpl <= 8 && seg.hist_len >= 8) return launch_interp<4, 8, 8>(seg, taps_host, stream);
        if (seg.interp == 2 && kpl <= 16 && seg.hist_len >= 16) return launch_interp<2, 16, 8>(seg, taps_host, stream);
        if (seg.interp == 8 && kpl <= 8 && seg.hist_len >= 8) return launch_interp<8, 8, 8>(seg, taps_host, stream);
    }
    return launch_generic(seg, taps_dev, stream);
}

}  // namespace cb
