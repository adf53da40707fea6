// K3-TC: polyphase interpolating FIR (zero-stuff xL then FIR, real or complex taps) as a Toeplitz GEMM
// on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM), sm_100a only.
//
// Reference semantics (src/pulse.rs:82-92, src/util/resample_node.rs:120-131 + src/filter/fir.rs:87-102):
//   y[L u + p] = sum_{j < TPP} h[L j + p] * x[u - j]          (the products with stuffed zeros dropped)
// BASELINE config 5 (L = 8, 1024 taps -> 128 taps per phase) needs 4096 real MACs per symbol per
// component pair; on the FP32 pipe that caps a B200 near 9 Gsym/s.  Here the MACs run on the
// tensor pipe and the kernel is bounded by the 64 B/symbol it has to write.
//
// Formulation.  RS = 128 / L symbols per stream row.  For one tile the symbol stream incl. HALO
// symbols of history, de-interleaved into a real and an imaginary fp16 stream S_c[e] (e = 0 ..
// 128 RS - 1), is stored ONCE, contiguously, in shared memory.  Read as a K-major matrix with a row
// pitch of RS elements (= the 32/64/128-byte swizzle row), row n of that buffer starts RS symbols
// after row n-1, so the buffer itself is the Toeplitz operand:
//     D[m][n] = sum_k H[m][k] * S_c[RS n + k],   k in [0, KT),  KT = 16 KS >= RS + TPP - 1
//     m = i L + p  (symbol i of the row, phase p)  ->  H[m][k] = h[L (i + HALO - k) + p]
// i.e. TMEM lane m holds output sample (128 n + m) of the tile: the 128 lanes of one column are 128
// CONSECUTIVE output samples, so the epilogue stores straight from registers, fully coalesced,
// with no shared-memory transpose.  The imaginary stream sits 128 rows after the real one, so a
// single N = 256 MMA (columns 0-127 real, 128-255 imaginary) covers both; the last
// ceil(KT/RS) - 1 columns of each half would read across the seam and are simply not used
// (VR valid rows per tile, 120 of 128 for config 5).  K step ks of the stream operand is the same
// buffer shifted by 32 ks bytes (descriptor start address only).
//
// Complex taps (CPLX): y = Hr*x + j Hi*x needs  D_re += Hr S_re - Hi S_im,  D_im += Hr S_im + Hi S_re.
// The stage holds a third region, -S_re, behind S_im, so that the same N = 256 operand shifted by one
// region is [S_im | -S_re]; with the image of -Hi as the M operand that one MMA adds exactly the two
// cross terms.  Twice the MMAs (54 per tile for config 5), same HBM traffic.
//
// Precision.  As in fir_tc_kernel.cu: stream and taps are block-scaled by exact powers of two into
// [2^14, 2^15) and split into fp16 hi + lo; three products (hi*hi, lo*hi, hi*lo) accumulate in the
// same fp32 TMEM accumulator.  Relative L2 error vs the sequential f32 form ~3e-7 (tolerance 1e-5).
//
// Roles (E epilogue warps first, E = 4, or 8 with the fused i16 quantiser; one persistent CTA per SM):
//   warps E..E+3 loaders / converters: raw f32 tile (coalesced LDG.128; or, with the fused quantiser, from a
//              ring of raw stages that the TMA warp E+5 fills with 4 KiB bulk copies one or two tiles ahead)
//              -> block max -> scale, split, de-interleave, st.shared (pre-swizzled) -> fence.proxy.async
//              -> mbarrier a_full
//   warp  E+4  one thread issues 3 KS tcgen05.mma (M128 N256 K16) per tile, commits a_empty/t_full
//   warps 0..E-1 epilogue (E/4 per TMEM sub-partition, alternating 32-column chunks): tcgen05.ld 32 lanes
//              x 32 columns (re) + (im) -> unscale [-> i16] -> st.global
// Two stream stages and two TMEM accumulator stages (2 x 256 columns) overlap the roles.
// Algorithmic HBM traffic: 8 B read + 8 L B written per symbol.
#include <cuda_fp16.h>

#include <vector>

#include "fir_kernels.cuh"

namespace cb {

namespace ptc {

// epilogue warps: warp w drains TMEM sub-partition w % 4, 32-column chunks w / 4, w / 4 + NEPI / 4, ...
// 4 are enough for f32 output; the fused i16 quantiser doubles the per-column work and gets 8
__host__ __device__ constexpr int nepi(bool out16) { return out16 ? 8 : 4; }
// + 4 loader / converter warps + MMA warp (+ TMA warp when the raw tile is staged by bulk copies)
__host__ __device__ constexpr int nthreads(bool out16) { return 32 * (nepi(out16) + 4 + (out16 ? 2 : 1)); }
constexpr int NLOAD = 128;                    // loader threads

struct Args {
    const float2 *x;
    const float2 *halo;     // HALO symbols preceding x[0] (16-byte aligned)
    float2 *y;
    const float2 *hist_in;
    float2 *hist_out;
    const uint4 *himg;      // prepacked tap image: [Hr hi, Hr lo (, -Hi hi, -Hi lo)][KS][128 rows x 32 B], 32-byte swizzled
    unsigned long long n;   // input symbols
    unsigned hist_len;
    unsigned ks;            // K steps of 16
    float tap_inv_scale;
    int2 *y16;              // OUT16: interleaved i16 IQ output (src/io/raw_iq.rs layout) instead of y
    float qscale;           // OUT16: (qscale * v) as i16, truncating, saturating
    unsigned *fix_count;    // tiles flagged for the exact fall-back pass (FirFix), or NULL
    unsigned *fix_list;
};

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred P;\n"
        "elect.sync _|P, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, P;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t *r)
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major swizzled shared-memory matrix descriptor.  ROWB = swizzle row bytes (32 / 64 / 128); the
// 8-row groups are 8 ROWB apart.  The swizzle XOR acts on absolute shared-memory address bits, so
// a start address shifted by whole rows or 32-byte K steps needs no base-offset field.
template <int ROWB>
__device__ __forceinline__ uint64_t kdesc(uint32_t saddr)
{
    constexpr uint64_t LAYOUT = ROWB == 128 ? 2 : (ROWB == 64 ? 4 : 6);
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8 * ROWB) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= LAYOUT << 61;
    return d;
}

template <int ROWB>
__host__ __device__ __forceinline__ uint32_t swz(uint32_t o)
{
    return o ^ (((o >> 7) & (uint32_t)(ROWB / 16 - 1)) << 4);
}

template <int L, bool CPLX>
struct Geo {
    static constexpr int RS = 128 / L;                 // symbols per stream row
    static constexpr int ROWB = 2 * RS;                // swizzle row bytes
    static constexpr int NEL = 128 * RS;               // stream elements per component per tile
    static constexpr int COMP = 128 * ROWB;            // bytes per component region
    static constexpr int NREG = CPLX ? 3 : 2;          // regions: re, im (, -re)
    static constexpr int PART = NREG * COMP + 1024;    // hi (or lo) part: regions + zeroed tail pad
    static constexpr int STAGE = 2 * PART;
    static constexpr int NLD = NEL / 2 / NLOAD;        // float4 loads per loader thread per tile
};

// Rust `v as i16` of a float: truncate toward zero, saturate, NaN -> 0 (examples/single_thread_bpsk.rs:40-48): one F2I
// (saturating to s32, NaN -> 0) and an integer clamp.  An ALU-only form (clamp, add 2^23 to |v| toward zero, restore
// the sign: 9 full-rate instructions instead of 3) was faster while the epilogue had 4 warps and its conversions
// queued on the quarter-rate pipe; with 8 epilogue warps the kernel is short of issue slots instead and the F2I form
// takes pulse4_i16 from 0.389 to 0.298 ms (63 -> 83 % of its 24 B/symbol roof).
__device__ __forceinline__ uint32_t trunc_i16(float v)
{
    const int q = __float2int_rz(v);
    return (uint32_t)min(max(q, -32768), 32767) & 0xFFFFu;
}

// OUT16: the example's quantiser `(8192 x) as i16` fused into the epilogue: 4 bytes written per output
// sample instead of 8 (and no separate pass over the f32 result)
// Raw tile supply, measured both ways on config 1: with f32 output the kernel is HBM-bound (96 % of the roof) and
// per-thread LDG.128 loads straight into registers are best; with the i16 output the write traffic halves, the
// exposed load latency of the single loader group becomes the limiter, and a TMA warp that keeps a ring of NRAW
// raw tiles filled ahead of the converters wins (0.436 -> 0.398 ms).  TMA_LOAD = OUT16.
// SMIN: the quiet test per symbol (taps that may skip one symbol of every pair, FirTcPlan::sample_min)
template <int L, bool CPLX, bool OUT16, int NRAW, bool SMIN>
__global__ void __launch_bounds__(OUT16 ? 512 : 288, 1) fir_ptc_kernel(const __grid_constant__ Args a)  // 512: 128-register cap (14 warps)
{
    constexpr bool TMA_LOAD = OUT16;
    constexpr int NEPI = nepi(OUT16), NTHREADS = nthreads(OUT16);
    constexpr int RAWB = Geo<L, CPLX>::NEL * 8;  // bytes of one raw tile (incl. halo)
    using G = Geo<L, CPLX>;
    constexpr int RS = G::RS, ROWB = G::ROWB, NLD = G::NLD;
    constexpr uint32_t IDESC = (1u << 4) | ((256u >> 3) << 17) | ((128u >> 4) << 24);  // f16 x f16 -> f32, M128 N256

    const int KS = (int)a.ks;
    const int KT = 16 * KS;
    const int HALO = KT - RS;                    // history symbols per tile
    const int VR = (G::NEL - KT) / RS + 1;       // valid stream rows (columns of D) per tile
    const int TS = VR * RS;                      // symbols per tile

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char *sS = smem;                            // 2 stages x (hi, lo)
    unsigned char *sH = smem + 2 * G::STAGE;             // tap image: KS*4096 bytes per part
    unsigned char *sRaw = sH + KS * (CPLX ? 16384 : 8192);  // NRAW raw f32 tiles
    __shared__ __align__(8) uint64_t a_full[2], a_empty[2], t_full[2], t_empty[2], sc_ready[8];
    __shared__ __align__(8) uint64_t raw_full[NRAW], raw_empty[NRAW];
    __shared__ uint32_t tmem_slot;
    __shared__ float red_max[4];
    __shared__ uint32_t red_min[4];
    __shared__ unsigned fix_seen;  // tile + 1 last appended to the fix-up list
    __shared__ float inv_scale[8];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned long long ntiles = (a.n + (unsigned long long)TS - 1) / (unsigned long long)TS;

    if (tid == 0) {
        fix_seen = 0u;
        for (int i = 0; i < 2; ++i) {
            mbar_init(&a_full[i], NLOAD);
            mbar_init(&a_empty[i], 1);
            mbar_init(&t_full[i], 1);
            mbar_init(&t_empty[i], 32 * NEPI);
        }
        for (int i = 0; i < 8; ++i) mbar_init(&sc_ready[i], 1);
        for (int i = 0; i < NRAW; ++i) {
            mbar_init(&raw_full[i], 1);
            mbar_init(&raw_empty[i], NLOAD);
        }
        fence_mbar_init();
    }
    if (warp == NEPI + 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)),
                     "r"(512)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // tap image -> shared; zero the tail pads the (unused) seam columns read
    for (int i = tid; i < KS * (CPLX ? 16384 : 8192) / 16; i += NTHREADS) reinterpret_cast<uint4 *>(sH)[i] = a.himg[i];
    for (int i = tid; i < 4 * 1024 / 16; i += NTHREADS) {
        const int part = i >> 6, o = i & 63;
        reinterpret_cast<uint4 *>(sS + part * G::PART + G::NREG * G::COMP)[o] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (TMA_LOAD)
        for (int i = tid; i < NRAW * RAWB / 16; i += NTHREADS) reinterpret_cast<uint4 *>(sRaw)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (TMA_LOAD && warp == NEPI + 5) {
        // ------------------------------------------------------------------ TMA producer: raw f32 tiles, HBM -> shared
        // tile elements e = 0 .. NEL-1 are symbols g = t0 - HALO + e: the first tile's halo comes from the history
        // buffer, everything else from x; an odd trailing sample (16-byte granularity) is left to the converters
        unsigned long long it = 0;
        const uint64_t pol = l2_evict_first_policy();
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int rs = (int)(it % NRAW);
            const uint32_t ph = (uint32_t)((it / NRAW) & 1);
            const long long g0 = (long long)tile * TS - HALO;
            const long long g_lo = g0 < 0 ? 0 : g0;
            long long g_hi = g0 + G::NEL;
            if (g_hi > (long long)a.n) g_hi = (long long)a.n & ~1ll;
            if (g_hi < g_lo) g_hi = g_lo;
            mbar_wait_long(&raw_empty[rs], ph ^ 1);
            unsigned char *dstb = sRaw + rs * RAWB;
            if (lane == 0) mbar_arrive_expect_tx(&raw_full[rs], (uint32_t)((g_hi - g_lo) * 8 + (g0 < 0 ? -g0 * 8 : 0)));
            __syncwarp();
            if (g0 < 0 && lane == 31) tma_load_1d(dstb, a.halo + (HALO + g0), (uint32_t)(-g0 * 8), &raw_full[rs]);
            for (long long g = g_lo + (long long)lane * 512; g < g_hi; g += 32 * 512) {  // 4 KiB pieces
                const long long n = g_hi - g < 512 ? g_hi - g : 512;
                tma_load_1d_hint(dstb + (g - g0) * 8, a.x + g, (uint32_t)(n * 8), &raw_full[rs], pol);
            }
        }
    } else if (warp >= NEPI && warp < NEPI + 4) {
        // ------------------------------------------------------------------ converters (block scale, fp16 split)
        const int gt = tid - 32 * NEPI, gw = warp - NEPI;
        if (a.hist_out != nullptr && blockIdx.x == 0) {
            const long long H = a.hist_len;
            for (long long i = gt; i < H; i += NLOAD) {
                const long long g = (long long)a.n - H + i;
                a.hist_out[i] = g >= 0 ? a.x[g] : a.hist_in[H + g];
            }
        }
        unsigned long long it = 0;
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = (int)(it & 1);
            const uint32_t ph = (uint32_t)((it >> 1) & 1);
            const long long t0 = (long long)tile * TS;
            const int rs = (int)(it % NRAW);
            float4 raw[NLD];
            float mx = 0.f;            // tile maximum
            uint32_t mnu = 0xffffffffu;  // bits of the smallest non-zero pair maximum, minus one (a zero pair wraps to the top)
            if (TMA_LOAD) mbar_wait(&raw_full[rs], (uint32_t)((it / NRAW) & 1));
            const float4 *rawt = reinterpret_cast<const float4 *>(sRaw + rs * RAWB);
#pragma unroll
            for (int i = 0; i < NLD; ++i) {
                const int q = gt + i * NLOAD;               // pair index: elements 2q, 2q+1
                const long long g = t0 - HALO + 2 * q;      // even
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (g < 0 || g + 1 < (long long)a.n) {
                    if (TMA_LOAD) v = rawt[q];
                    else v = ldg_stream(reinterpret_cast<const float4 *>(g < 0 ? a.halo + (HALO + g) : a.x + g));
                } else if (g < (long long)a.n) {            // odd trailing sample (not covered by 16-byte copies)
                    const float2 t = a.x[g];
                    v = make_float4(t.x, t.y, 0.f, 0.f);
                }
                raw[i] = v;
                const float pm = fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));
                mx = fmaxf(mx, pm);
                mnu = min(mnu, quiet_key<SMIN>(v, pm));
            }
            if (TMA_LOAD) mbar_arrive(&raw_empty[rs]);  // the raw tile is in registers: the TMA warp may refill the stage
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                mnu = min(mnu, __shfl_xor_sync(0xffffffffu, mnu, o));
            }
            if (lane == 0) {
                red_max[gw] = mx;
                red_min[gw] = mnu;
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mx = fmaxf(fmaxf(red_max[0], red_max[1]), fmaxf(red_max[2], red_max[3]));
            mnu = min(min(red_min[0], red_min[1]), min(red_min[2], red_min[3]));
            asm volatile("bar.sync 1, 128;" ::: "memory");  // red_max / red_min are reused by the next tile
            // quiet stretch more than 2^20 below the tile maximum: recomputed in plain f32 by the fix-up pass (FirFix,
            // fir_kernels.cuh); non-finite symbols are caught in the conversion loop below
            if (gt == 0 && a.fix_count != nullptr && mnu != 0xffffffffu && __uint_as_float(mnu + 1u) < mx * 9.5367431640625e-7f &&
                atomicExch(&fix_seen, (unsigned)tile + 1u) != (unsigned)tile + 1u)
                a.fix_list[atomicAdd(a.fix_count, 1u)] = (unsigned)tile;
            uint32_t eb = (__float_as_uint(mx) >> 23) & 0xFF;
            eb = (eb < 16 || eb == 255) ? 141 : eb;  // all-zero / denormal / non-finite tile: scale 1
            const float sc = __uint_as_float((268u - eb) << 23);
            if (gt == 0) {  // the epilogue is at most 4 tiles behind: an 8-deep ring cannot wrap
                inv_scale[it & 7] = __uint_as_float((eb - 14u) << 23);
                mbar_arrive(&sc_ready[it & 7]);
            }
            mbar_wait(&a_empty[s], ph ^ 1);  // the MMAs that read this stage two tiles ago are done
            unsigned char *hi = sS + s * G::STAGE, *lo = hi + G::PART;
            __half2 nanacc = __floats2half2_rn(0.f, 0.f);  // sum of the lo terms: NaN iff a symbol of the tile is Inf / NaN
#pragma unroll
            for (int i = 0; i < NLD; ++i) {
                const int q = gt + i * NLOAD;
                const float4 v = make_float4(raw[i].x * sc, raw[i].y * sc, raw[i].z * sc, raw[i].w * sc);
                const __half2 hr = __floats2half2_rn(v.x, v.z), hm = __floats2half2_rn(v.y, v.w);  // (re0,re1), (im0,im1)
                const float2 br = __half22float2(hr), bm = __half22float2(hm);
                const __half2 lr = __floats2half2_rn(v.x - br.x, v.z - br.y);
                const __half2 lm = __floats2half2_rn(v.y - bm.x, v.w - bm.y);
                nanacc = __hadd2(nanacc, __hadd2(lr, lm));  // Inf * sc - Inf = NaN, NaN stays NaN; finite |lo| < 16
                const uint32_t off = swz<ROWB>((uint32_t)q * 4u);
                *reinterpret_cast<__half2 *>(hi + off) = hr;
                *reinterpret_cast<__half2 *>(hi + G::COMP + off) = hm;
                *reinterpret_cast<__half2 *>(lo + off) = lr;
                *reinterpret_cast<__half2 *>(lo + G::COMP + off) = lm;
                if (CPLX) {  // third region: -re
                    *reinterpret_cast<__half2 *>(hi + 2 * G::COMP + off) = __hneg2(hr);
                    *reinterpret_cast<__half2 *>(lo + 2 * G::COMP + off) = __hneg2(lr);
                }
            }
            fence_proxy_async();
            mbar_arrive(&a_full[s]);
            if (a.fix_count != nullptr && (__hisnan(__low2half(nanacc)) || __hisnan(__high2half(nanacc))) &&
                atomicExch(&fix_seen, (unsigned)tile + 1u) != (unsigned)tile + 1u)
                a.fix_list[atomicAdd(a.fix_count, 1u)] = (unsigned)tile;  // non-finite symbol: exact fall-back (FirFix)
        }
    } else if (warp == NEPI + 4) {
        // ------------------------------------------------------------------ MMA issuer
        // The whole warp runs the loop, one elected lane issues: warp-uniform code keeps the descriptors in uniform
        // registers (base descriptor + (byte offset >> 4)); inside `if (lane == 0)` every tcgen05.mma was wrapped in an
        // ELECT / R2UR.BROADCAST / branch sequence.
        unsigned long long it = 0;
        const uint64_t hd0 = kdesc<32>(smem_u32(sH)), sd0 = kdesc<ROWB>(smem_u32(sS));
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = (int)(it & 1);
            const uint32_t ph = (uint32_t)((it >> 1) & 1);
            mbar_wait_long(&t_empty[s], ph ^ 1);
            mbar_wait_long(&a_full[s], ph);
            tc_fence_after();
            const uint64_t shi = sd0 + (uint64_t)((s * G::STAGE) >> 4), slo = shi + (uint64_t)(G::PART >> 4);
            const uint64_t hlo = hd0 + (uint64_t)((KS * 4096) >> 4);
            const uint32_t d = tmem_base + (uint32_t)s * 256u;
            if (elect_one()) {
                for (int ks = 0; ks < KS; ++ks) {
                    const uint64_t ah = hd0 + (uint64_t)(ks * 256);          // ks * 4096 bytes
                    const uint64_t al = hlo + (uint64_t)(ks * 256);
                    const uint64_t bh = shi + (uint64_t)(ks * 2);            // ks * 32 bytes
                    const uint64_t bl = slo + (uint64_t)(ks * 2);
                    tc_mma(d, ah, bh, IDESC, ks > 0 ? 1u : 0u);
                    tc_mma(d, al, bh, IDESC, 1u);
                    tc_mma(d, ah, bl, IDESC, 1u);
                    if (CPLX) {  // (-Hi) x [S_im | -S_re]
                        const uint64_t ch = hd0 + (uint64_t)((2 * KS + ks) * 256);
                        const uint64_t cl = hd0 + (uint64_t)((3 * KS + ks) * 256);
                        const uint64_t dh = shi + (uint64_t)((G::COMP >> 4) + ks * 2);
                        const uint64_t dl = slo + (uint64_t)((G::COMP >> 4) + ks * 2);
                        tc_mma(d, ch, dh, IDESC, 1u);
                        tc_mma(d, cl, dh, IDESC, 1u);
                        tc_mma(d, ch, dl, IDESC, 1u);
                    }
                }
                tc_commit(&a_empty[s]);
                tc_commit(&t_full[s]);
            }
            __syncwarp();
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 0 .. NEPI-1)
        const int e = warp & 3;  // TMEM sub-partition = warp % 4; lane m = 32 e + lane
        const int m = 32 * e + lane;
        const int msym = m / L;
        unsigned long long it = 0;
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = (int)(it & 1);
            const uint32_t ph = (uint32_t)((it >> 1) & 1);
            const long long t0 = (long long)tile * TS;
            mbar_wait(&sc_ready[it & 7], (uint32_t)((it >> 3) & 1));
            const float k = inv_scale[it & 7] * a.tap_inv_scale;  // a power of two
            // OUT16: (qscale * (acc * k)) as i16.  When qscale is a power of two as well (8192 in the examples)
            // the two roundings collapse into one exact product; otherwise both multiplies are kept so that the
            // result equals quantising the f32 output.
            const bool q_pow2 = OUT16 && (__float_as_uint(a.qscale) & 0x007FFFFFu) == 0u && a.qscale > 0.f;
            const float kq = q_pow2 ? k * a.qscale : k;
            mbar_wait_long(&t_full[s], ph);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * e) << 16) + (uint32_t)s * 256u;
            float2 *yrow = a.y + (long long)L * t0 + m;   // + 128 n per column
            uint32_t *qrow = reinterpret_cast<uint32_t *>(a.y16) + (long long)L * t0 + m;
            // columns n < nlive are stored: n < VR and symbol t0 + RS n + msym < a.n
            const long long srem = (long long)a.n - t0 - msym;
            const int nlive = srem <= 0 ? 0 : (srem >= (long long)RS * VR ? VR : (int)((srem + RS - 1) / RS));
#pragma unroll 1
            for (int c = warp >> 2; c < 4; c += NEPI / 4) {
                if (32 * c >= VR) break;
                uint32_t p[32], r[32];
                tc_ld32(taddr + 32 * c, p);
                tc_ld32(taddr + 128 + 32 * c, r);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int n = 32 * c + j;
                    // values are formed unconditionally (branch-free body: the 32 columns interleave in the
                    // schedule); only the store is predicated
                    const bool live = n < nlive;
                    if (OUT16) {
                        float vx = __uint_as_float(p[j]) * kq, vy = __uint_as_float(r[j]) * kq;
                        if (!q_pow2) {
                            vx = __fmul_rn(a.qscale, vx);
                            vy = __fmul_rn(a.qscale, vy);
                        }
                        const uint32_t q = trunc_i16(vx) | (trunc_i16(vy) << 16);
                        if (live) qrow[128 * n] = q;
                    } else {
                        const float2 v = make_float2(__uint_as_float(p[j]) * k, __uint_as_float(r[j]) * k);
                        if (live) stg_stream2(yrow + 128 * n, v);
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(&t_empty[s]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == NEPI + 4) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

}  // namespace ptc

// ------------------------------------------------------------------------------------ host side
static int ptc_rs(uint32_t L) { return 128 / (int)L; }

int fir_ptc_ksteps(uint32_t ntaps, uint32_t L)
{
    const int tpp = (int)ceil_div(ntaps ? ntaps : 1, (size_t)L);
    return (int)ceil_div((size_t)(ptc_rs(L) + tpp - 1), (size_t)16);
}

bool fir_ptc_supported(uint32_t ntaps, uint32_t L, bool taps_real)
{
    if (ntaps == 0 || (L != 8 && L != 4)) return false;
    const int ks = fir_ptc_ksteps(ntaps, L);
    if (ks < 1 || ks > 12) return false;
    // shared memory: two stream stages + the tap image (+ alignment slack) must fit in 227 KiB
    const size_t comp = (size_t)128 * 2 * ptc_rs(L);
    const size_t stage = 2 * ((taps_real ? 2 : 3) * comp + 1024);
    const size_t raw = (size_t)128 * ptc_rs(L) * 8;  // one raw f32 tile
    return 2 * stage + fir_ptc_image_bytes(ntaps, L, taps_real) + raw + 1024 <= 227 * 1024;
}

size_t fir_ptc_image_bytes(uint32_t ntaps, uint32_t L, bool taps_real)
{
    return (size_t)fir_ptc_ksteps(ntaps, L) * (taps_real ? 8192 : 16384);
}

// Tap image: part (Hr hi, Hr lo[, -Hi hi, -Hi lo]) x K step x [128 rows x 32 bytes], 32-byte swizzled, fp16.
void fir_ptc_build_image(const float2 *taps, uint32_t ntaps, uint32_t L, bool taps_real, unsigned char *img,
                         float *tap_inv_scale)
{
    const int KS = fir_ptc_ksteps(ntaps, L);
    const int RS = ptc_rs(L), KT = 16 * KS, HALO = KT - RS;
    float mx = 0.f;
    for (uint32_t k = 0; k < ntaps; ++k) mx = fmaxf(mx, fmaxf(fabsf(taps[k].x), fabsf(taps[k].y)));
    uint32_t bits;
    memcpy(&bits, &mx, 4);
    uint32_t eb = (bits >> 23) & 0xFF;
    if (eb < 16 || eb == 255) eb = 141;
    const uint32_t sb = (268u - eb) << 23, ib = (eb - 14u) << 23;
    float sc;
    memcpy(&sc, &sb, 4);
    memcpy(tap_inv_scale, &ib, 4);
    memset(img, 0, fir_ptc_image_bytes(ntaps, L, taps_real));
    for (int c = 0; c < (taps_real ? 1 : 2); ++c) {
        for (int m = 0; m < 128; ++m) {
            const int i = m / (int)L, p = m % (int)L;
            for (int k = 0; k < KT; ++k) {
                const long long t = (long long)L * (i + HALO - k) + p;
                float v = 0.f;
                if (i + HALO - k >= 0 && t < (long long)ntaps) v = c == 0 ? taps[t].x : -taps[t].y;
                v *= sc;
                const __half h = __float2half_rn(v);
                const __half l = __float2half_rn(v - __half2float(h));
                const int ks = k >> 4, kk = k & 15;
                const uint32_t o = ptc::swz<32>((uint32_t)m * 32u + (uint32_t)kk * 2u);
                memcpy(img + (size_t)(2 * c * KS + ks) * 4096 + o, &h, 2);
                memcpy(img + (size_t)((2 * c + 1) * KS + ks) * 4096 + o, &l, 2);
            }
        }
    }
}

template <int L, bool CPLX, bool OUT16, int NRAW, bool SMIN>
static int launch_ptc_raw(const ptc::Args &a, cudaStream_t stream)
{
    using G = ptc::Geo<L, CPLX>;
    const int SMEM = 2 * G::STAGE + (int)a.ks * (CPLX ? 16384 : 8192) + (OUT16 ? NRAW * G::NEL * 8 : 0) + 1024;
    auto kern = ptc::fir_ptc_kernel<L, CPLX, OUT16, NRAW, SMIN>;
    CB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    const int KT = 16 * (int)a.ks;
    const unsigned long long TS = (unsigned long long)(((G::NEL - KT) / G::RS + 1) * G::RS);
    const unsigned long long ntiles = (a.n + TS - 1) / TS;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned grid = (unsigned)(ntiles < (unsigned long long)sms ? ntiles : (unsigned long long)sms);
    kern<<<grid, ptc::nthreads(OUT16), SMEM, stream>>>(a);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

// two raw stages when they fit in shared memory, else one
template <int L, bool CPLX, bool OUT16>
static int launch_ptc_l(const ptc::Args &a, bool smin, cudaStream_t stream)
{
    using G = ptc::Geo<L, CPLX>;
    const size_t need2 = 2 * (size_t)G::STAGE + (size_t)a.ks * (CPLX ? 16384 : 8192) + 2 * (size_t)G::NEL * 8 + 1024;
    if (!OUT16 || need2 <= 227 * 1024)
        return smin ? launch_ptc_raw<L, CPLX, OUT16, 2, true>(a, stream) : launch_ptc_raw<L, CPLX, OUT16, 2, false>(a, stream);
    return smin ? launch_ptc_raw<L, CPLX, OUT16, 1, true>(a, stream) : launch_ptc_raw<L, CPLX, OUT16, 1, false>(a, stream);
}

bool fir_ptc_applicable(const FirSeg &seg, bool taps_real)
{
    if (seg.decim != 1 || !fir_ptc_supported(seg.ntaps, seg.interp, taps_real)) return false;
    const uint32_t halo = 16u * (uint32_t)fir_ptc_ksteps(seg.ntaps, seg.interp) - (uint32_t)ptc_rs(seg.interp);
    if (seg.hist_len < halo) return false;
    const float2 *h = seg.hist_in + (seg.hist_len - halo);
    return ((reinterpret_cast<uintptr_t>(seg.x) | reinterpret_cast<uintptr_t>(h)) & 15) == 0 &&
           (reinterpret_cast<uintptr_t>(seg.y) & 7) == 0 && (reinterpret_cast<uintptr_t>(seg.y16) & 3) == 0;
}

// symbols per tile of the kernel above (TS in fir_ptc_kernel)
static unsigned ptc_tile_symbols(uint32_t interp, unsigned ks)
{
    const int rs = 128 / (int)interp, nel = 128 * rs, kt = 16 * (int)ks;
    return (unsigned)(((nel - kt) / rs + 1) * rs);
}

static int launch_fir_ptc_main(const FirSeg &seg, const ptc::Args &a, bool taps_real, bool smin, cudaStream_t stream);

int launch_fir_ptc(const FirSeg &seg, const FirTcPlan &plan, bool taps_real, const float2 *taps_dev, cudaStream_t stream)
{
    FirFix *fix = plan.fix;
    if (seg.n_in == 0) return CB_OK;
    ptc::Args a;
    a.ks = (unsigned)fir_ptc_ksteps(seg.ntaps, seg.interp);
    a.x = seg.x;
    a.halo = seg.hist_in + (seg.hist_len - (16u * a.ks - (uint32_t)ptc_rs(seg.interp)));
    a.y = seg.y;
    a.hist_in = seg.hist_in;
    a.hist_out = seg.hist_out;
    a.himg = reinterpret_cast<const uint4 *>(plan.bimg_dev);
    a.n = seg.n_in;
    a.hist_len = seg.hist_len;
    a.tap_inv_scale = plan.tap_inv_scale;
    a.y16 = reinterpret_cast<int2 *>(seg.y16);
    a.qscale = seg.qscale;
    const unsigned ts = ptc_tile_symbols(seg.interp, a.ks);
    const bool fixup = fix != nullptr && fix->dev != nullptr && taps_dev != nullptr && fix->cap >= ceil_div(seg.n_in, (size_t)ts);
    a.fix_count = fixup ? fix->dev + (fix->calls & 1u) : nullptr;
    a.fix_list = fixup ? fix->dev + 2 : nullptr;
    const int rc = launch_fir_ptc_main(seg, a, taps_real, plan.sample_min, stream);
    if (rc || !fixup) return rc;
    FirFixArgs f{seg.x, seg.hist_in, taps_dev, seg.y, seg.y16, seg.qscale, seg.n_in, seg.ntaps, seg.interp, ts, seg.hist_len,
                 a.fix_count, fix->dev + ((fix->calls + 1) & 1u), a.fix_list};
    ++fix->calls;
    return launch_fir_fixup(f, stream);
}

static int launch_fir_ptc_main(const FirSeg &seg, const ptc::Args &a, bool taps_real, bool smin, cudaStream_t stream)
{
    if (seg.y16 != nullptr) {
        switch (seg.interp) {
        case 8: return taps_real ? launch_ptc_l<8, false, true>(a, smin, stream) : launch_ptc_l<8, true, true>(a, smin, stream);
        case 4: return taps_real ? launch_ptc_l<4, false, true>(a, smin, stream) : launch_ptc_l<4, true, true>(a, smin, stream);
        default: break;
        }
    }
    switch (seg.interp) {
    case 8: return taps_real ? launch_ptc_l<8, false, false>(a, smin, stream) : launch_ptc_l<8, true, false>(a, smin, stream);
    case 4: return taps_real ? launch_ptc_l<4, false, false>(a, smin, stream) : launch_ptc_l<4, true, false>(a, smin, stream);
    default: set_error("fir_ptc: unsupported interpolation factor %u", seg.interp); return CB_ERR_UNSUPPORTED;
    }
}

}  // namespace cb
