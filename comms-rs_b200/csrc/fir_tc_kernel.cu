// K1-TC: complex FIR (decim = interp = 1, up to 128 taps) as a block-Toeplitz GEMM on the
// 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM), sm_100a only.
//
// Reference semantics (src/filter/fir.rs:87-102): y[n] = sum_{k<K} h[k] x[n-k], complex f32.
// In direct form the 64-tap complex filter costs 256 FP32 FMAs per sample, which caps the CUDA
// core kernel at ~35 % of the HBM roofline; here the MACs run on the tensor pipe instead.
//
// Formulation.  A tile is 128 rows x 32 complex outputs.  With S[p] = x[t0 - HALO + p] (the
// tile's input stream incl. halo, HALO = 32*(KB-1) >= taps) viewed as interleaved reals,
//     D[m][n] = sum_k A[m][k] * B[n][k],   A[m][k] = S~[64 m + k],   k in [0, 64 KB)
// where n = 2 i + c enumerates (output i, re/im) of the row and B is the real-ified Toeplitz tap
// matrix  B[2i+c][2j+d] = { hr, -hi ; hi, hr }[c][d] of tap t = i + HALO - j  (0 outside 0..K-1).
// Row m of A starts 64 reals = 128 bytes (fp16) after row m-1: the stream itself, stored once in
// shared memory in the 128-byte-swizzled K-major UMMA layout, IS the Toeplitz operand -- K-block
// kb of row m is just row m+kb of the same buffer (descriptor start address + 128*kb bytes).
//
// Precision.  fp16 operands alone would give ~1e-3; x and h are each split into two fp16 terms
// (hi + lo, after an exact power-of-two block scaling of the tile / of the taps into [2^14, 2^15)),
// and three products are accumulated in fp32:  A_hi*B_hi + A_hi*B_lo + A_lo*B_hi  (the lo*lo
// term is < 2^-22 relative).  A_hi * [B_hi ; B_lo] is one N=128 MMA (columns 0-63 / 64-127 of
// the accumulator), A_lo * B_hi one N=64 MMA into columns 0-63; the epilogue adds the halves.
// Relative L2 error against the f32 sequential form ~3e-7 (tolerance 1e-5).
//
// Roles (576 threads, one persistent CTA per SM, tiles round-robin):
//   warp  17     TMA producer: the raw tile (f32, or i16 IQ words with IQ16) HBM -> shared by bulk copies, NRAW stages
//   warps 0-5 / 6-11  two converter groups, even / odd tiles of the CTA, each feeding its own A stage:
//              raw tile -> registers (IQ16: widened there) -> block max -> exact power-of-two scale, hi / lo split,
//              st.shared (pre-swizzled) -> fence.proxy.async -> mbarrier a_full; tiles whose quiet stretches or
//              non-finite samples the two-term split cannot carry are appended to the exact fall-back's list
//   warp  16     the whole warp runs the loop, one elected lane issues 4*KB x 2 tcgen05.mma per tile,
//              tcgen05.commit -> a_empty, t_full
//   warps 12-15  epilogue: tcgen05.ld (32 lanes x 32 columns) -> add halves, unscale -> 256-bit streaming stores
//              (IQ16: (out_scale * y) as i16, packed words); a padded shared staging path for unaligned outputs
// Two A stages and two TMEM accumulator stages keep the roles overlapped; the copies of the next tiles are in flight
// while a tile is converted.  scripts/ftc_timeline.cu prints where every role's cycles go
// (profiles/r03x_fir_tc_phases.txt).
// Algorithmic HBM traffic: 8 B read + 8 B written per sample (IQ16: 4 + 4); the halo re-read is 1.5 %.
#include <cuda_fp16.h>

#include <vector>

#include "fir_kernels.cuh"

namespace cb {

namespace tc {

constexpr int ROWS = 128;          // MMA M
constexpr int RS = 32;             // complex outputs per row
constexpr int TILE = ROWS * RS;    // 4096 outputs per tile
constexpr int NCW = 6;             // warps per converter group
constexpr int NCONV = 32 * NCW;    // converter threads per group.  The groups' serial chain (wait raw tile -> max / min
                                   // reduction -> barrier -> scale, split, store) bounds the kernel; six warps instead of
                                   // four shorten it by a third (11 instead of 17 sample pairs per thread and tile)
constexpr int W_EPI = 2 * NCW;     // first of the 4 epilogue warps (a multiple of 4: TMEM sub-partition = warp % 4)
constexpr int W_MMA = W_EPI + 4, W_TMA = W_EPI + 5;
constexpr int NTHREADS = 32 * (W_TMA + 1);  // 2 converter groups + 4 epilogue warps + MMA warp + TMA warp
static_assert(W_EPI % 4 == 0, "epilogue warp w must own TMEM sub-partition w % 4");
constexpr int A_PART = 18432;      // bytes reserved for one fp16 stream part (>= (128+4)*128, 1024-aligned)
constexpr int A_STAGE = 2 * A_PART;
constexpr int OUT_PITCH = 272;     // padded row pitch of the output staging (bytes)
constexpr int OUT_WARP = 32 * OUT_PITCH;

struct Args {
    const float2 *x;
    const float2 *halo;     // HALO samples preceding x[0] (16-byte aligned)
    float2 *y;
    const float2 *hist_in;
    float2 *hist_out;
    const uint4 *bimg;      // prepacked B image, KB * 16384 bytes
    unsigned long long n;
    unsigned hist_len;
    float tap_inv_scale;    // 2^-(14 - e_h)
    unsigned *fix_count;    // tiles flagged for the exact fall-back pass (FirFix), or NULL
    unsigned *fix_list;
    // IQ16 (i16 IQ on both edges, src/io/raw_iq.rs:78-140, :185-223): one 32-bit word per sample
    const uint32_t *x16;    // input: x = in_scale * (i16 as f32), widened by the converter warps (x unused)
    uint32_t *y16;          // output: (out_scale * y) as i16, quantised by the epilogue warps (y unused)
    float in_scale, out_scale;
};

// Rust `as i16`: truncate toward zero, saturate, NaN -> 0 (misc_kernels.cu quant_i16).  One conversion-pipe instruction
// and a clamp per value: this epilogue is short of issue slots, not of conversion throughput
__device__ __forceinline__ int quant_i16(float v, float scale)
{
    const int q = __float2int_rz(__fmul_rn(scale, v));
    return min(max(q, -32768), 32767);
}
__device__ __forceinline__ uint32_t pack_i16(int lo, int hi) { return __byte_perm((uint32_t)lo, (uint32_t)hi, 0x5410); }
__device__ __forceinline__ float2 widen_iq16(uint32_t w, float scale)
{
    return make_float2(__fmul_rn(scale, (float)(int16_t)(w & 0xFFFFu)), __fmul_rn(scale, (float)(int16_t)(w >> 16)));
}

__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
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
// D[tmem] (+)= A[smem] * B[smem]^T, fp16 operands, fp32 accumulate.  One thread issues.
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
// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread
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

// K-major, 128-byte swizzle shared-memory matrix descriptor: 8-row groups 1024 bytes apart.
// The hardware applies the swizzle XOR to absolute shared-memory address bits, so a start address
// that is shifted by whole 128-byte rows (the Toeplitz trick) or by 32-byte K steps needs no
// base-offset field (measured: setting it to (addr >> 7) & 7 breaks the result).
__device__ __forceinline__ uint64_t tc_desc(uint32_t saddr)
{
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;             // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;   // stride byte offset
    d |= (uint64_t)1 << 46;             // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;             // SWIZZLE_128B
    return d;
}

__device__ __forceinline__ uint32_t swz128(uint32_t o) { return o ^ (((o >> 7) & 7) << 4); }

// NRAW raw f32 tiles are kept in flight by the TMA warp (2 when shared memory allows, i.e. up to 64 taps, else 1)
__device__ __noinline__ float4 iq16_edge_pair(const Args &a, long long g, int halo);

// scripts/ftc_timeline.cu compiles this file with CB_FTC_STATS: clock64 sums per phase of one thread of every role
#ifdef CB_FTC_STATS
__device__ unsigned long long *g_ftc_dbg = nullptr;
#define FTC_DECL unsigned long long st_[8] = {0}; long long t_ = clock64()
#define FTC_T(cond, k)                               \
    if (cond) {                                      \
        const long long now_ = clock64();            \
        st_[k] += (unsigned long long)(now_ - t_);   \
        t_ = now_;                                   \
    }
#define FTC_OUT(cond, role)                                                                            \
    if ((cond) && g_ftc_dbg != nullptr)                                                                \
        for (int k_ = 0; k_ < 8; ++k_) g_ftc_dbg[((size_t)blockIdx.x * 5 + (role)) * 8 + k_] = st_[k_]
#else
#define FTC_DECL
#define FTC_T(cond, k)
#define FTC_OUT(cond, role)
#endif

// IQ16: the raw tiles are i16 IQ words (half the bytes; the first tile's halo is read from the f32 history by the
// converters) and the epilogue writes i16 IQ words.  A tile of 16-bit samples never needs the exact fall-back, but the
// first one's halo can hold anything (set_state, an f32 call): that tile takes the quiet test of the f32 form, so the
// same tiles are recomputed and the words equal quantising the f32 result.
// SMIN: the quiet test per sample (taps that may skip one sample of every pair, FirTcPlan::sample_min).
template <int KB, int NRAW, bool IQ16 = false, bool SMIN = false>
__global__ void __launch_bounds__(NTHREADS, 1) fir_tc_kernel(const __grid_constant__ Args a)
{
    constexpr int HALO = RS * (KB - 1);            // complex samples of history per tile
    constexpr int NPAIR = (TILE + HALO) / 2;       // 16-byte pairs of complex samples per tile
    constexpr int NLD = (NPAIR + NCONV - 1) / NCONV;
    constexpr int B_BYTES = KB * 16384;
    constexpr uint32_t IDESC128 = (1u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
    constexpr uint32_t IDESC64 = (1u << 4) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // swizzle atoms need 1024 B
    unsigned char *sB = smem;                      // B image
    unsigned char *sA = smem + B_BYTES;            // 2 stages x (hi, lo)
    unsigned char *sOut = sA + 2 * A_STAGE;        // 4 warps x 32 rows x 272 B
    constexpr int RAWB = (TILE + HALO) * (IQ16 ? 4 : 8);  // one raw tile incl. halo
    unsigned char *sRaw = sOut + 4 * OUT_WARP;     // NRAW raw tiles (TMA destination)
    __shared__ __align__(8) uint64_t raw_full[NRAW], raw_empty[NRAW];
    __shared__ __align__(8) uint64_t a_full[2], a_empty[2], t_full[2], t_empty[2], sc_ready[8];
    __shared__ uint32_t tmem_slot;
    // [loader group][tile parity of the group][warp]: a warp that races ahead writes its next tile's partial result into
    // the other half, and cannot reach the tile after that before every warp of the group has passed the next
    // tile's barrier, i.e. has read this tile's values
    __shared__ float red_max[2][2][NCW];
    __shared__ uint32_t red_min[2][2][NCW];
    __shared__ unsigned fix_seen[2];  // tile + 1 last appended to the fix-up list by each converter group
    __shared__ float inv_scale[8];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned long long ntiles = (a.n + TILE - 1) / TILE;

    if (tid == 0) {
        fix_seen[0] = fix_seen[1] = 0u;
        for (int i = 0; i < 2; ++i) {
            mbar_init(&a_full[i], NCONV);
            mbar_init(&a_empty[i], 1);
            mbar_init(&t_full[i], 1);
            mbar_init(&t_empty[i], 128);
        }
        for (int i = 0; i < 8; ++i) mbar_init(&sc_ready[i], 1);
        for (int i = 0; i < NRAW; ++i) {
            mbar_init(&raw_full[i], 1);
            mbar_init(&raw_empty[i], NCONV);
        }
        fence_mbar_init();
    }
    if (warp == W_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)),
                     "r"(256)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // B image: plain copy, then publish to the async proxy (tcgen05.mma reads it)
    for (int i = tid; i < B_BYTES / 16; i += NTHREADS) reinterpret_cast<uint4 *>(sB)[i] = a.bimg[i];
    for (int i = tid; i < NRAW * RAWB / 16; i += NTHREADS) reinterpret_cast<uint4 *>(sRaw)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;

    if (warp == W_TMA) {
        // ------------------------------------------------------------------ TMA producer: raw f32 tiles, HBM -> shared
        // raw stage rs = it % NRAW holds samples g = t0 - HALO + e, e = 0 .. TILE + HALO - 1; the first tile's halo comes
        // from the history buffer; an odd trailing sample (16-byte copy granularity) is left to the converters
        unsigned long long it = 0;
        FTC_DECL;
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int rs = (int)(it % NRAW);
            const uint32_t ph = (uint32_t)((it / NRAW) & 1);
            const long long g0 = (long long)tile * TILE - HALO;
            const long long g_lo = g0 < 0 ? 0 : g0;
            long long g_hi = g0 + TILE + HALO;
            if (g_hi > (long long)a.n) g_hi = (long long)a.n & (IQ16 ? ~3ll : ~1ll);  // 16-byte copy granularity
            if (g_hi < g_lo) g_hi = g_lo;
            FTC_T(lane == 0, 0);
            mbar_wait_long(&raw_empty[rs], ph ^ 1);
            FTC_T(lane == 0, 1);
            unsigned char *dstb = sRaw + rs * RAWB;
            // 2 KiB pieces, one per lane.  (Issuing a bulk copy costs the warp ~100 cycles whatever its size and the
            // lanes' copies serialise: this warp is busy 1700 of a tile's 2800 cycles.  One 33 KiB copy per tile cuts the
            // tile to 2450 cycles -- and the SM clock under this kernel's load sags from 1.77 to 1.5 GHz, so the time
            // does not move: profiles/r03x_fir_tc_phases.txt.  Kept as pieces.)
            if constexpr (IQ16) {
                if (lane == 0) mbar_arrive_expect_tx(&raw_full[rs], (uint32_t)((g_hi - g_lo) * 4));
                __syncwarp();
                for (long long g = g_lo + (long long)lane * 512; g < g_hi; g += 32 * 512) {
                    const long long n = g_hi - g < 512 ? g_hi - g : 512;
                    tma_load_1d(dstb + (g - g0) * 4, a.x16 + g, (uint32_t)(n * 4), &raw_full[rs]);
                }
                continue;
            }
            if (lane == 0) mbar_arrive_expect_tx(&raw_full[rs], (uint32_t)((g_hi - g_lo) * 8 + (g0 < 0 ? -g0 * 8 : 0)));
            __syncwarp();
            if (g0 < 0 && lane == 31) tma_load_1d(dstb, a.halo + (HALO + g0), (uint32_t)(-g0 * 8), &raw_full[rs]);
            for (long long g = g_lo + (long long)lane * 256; g < g_hi; g += 32 * 256) {
                const long long n = g_hi - g < 256 ? g_hi - g : 256;
                tma_load_1d(dstb + (g - g0) * 8, a.x + g, (uint32_t)(n * 8), &raw_full[rs]);
            }
        }
        FTC_OUT(lane == 0, 0);
    } else if (warp < W_EPI) {
        // ------------------------------------------------------------------ converters (two groups, even / odd tiles)
        const int grp = warp / NCW, gt = tid - grp * NCONV, gw = warp - grp * NCW;
        if (a.hist_out != nullptr && blockIdx.x == 0 && grp == 0) {
            const long long H = a.hist_len;
            for (long long i = gt; i < H; i += NCONV) {
                const long long g = (long long)a.n - H + i;
                if constexpr (IQ16) a.hist_out[i] = g >= 0 ? widen_iq16(a.x16[g], a.in_scale) : a.hist_in[H + g];
                else a.hist_out[i] = g >= 0 ? a.x[g] : a.hist_in[H + g];
            }
        }
        unsigned long long it = grp;
        FTC_DECL;
        for (unsigned long long tile = blockIdx.x + (unsigned long long)grp * gridDim.x; tile < ntiles;
             tile += 2ull * gridDim.x, it += 2) {
            const int s = grp;
            const uint32_t ph = (uint32_t)((it >> 1) & 1);
            const long long t0 = (long long)tile * TILE;
            float4 raw[NLD];
            float mx = 0.f;            // tile maximum
            uint32_t mnu = 0xffffffffu;  // bits of the smallest non-zero pair maximum, minus one (a zero pair wraps to the top)
            const int rs = (int)(it % NRAW);
            FTC_T(gt == 0, 0);
            mbar_wait(&raw_full[rs], (uint32_t)((it / NRAW) & 1));
            FTC_T(gt == 0, 1);
            const float4 *rawt = reinterpret_cast<const float4 *>(sRaw + rs * RAWB);
            if constexpr (IQ16) {
                // all the tile's words first (NLD loads in flight), widened branch-free; the first tile's halo (f32
                // history) and the up to three trailing samples the 16-byte bulk copies leave out are patched afterwards,
                // out of line, so that the loop every tile runs stays small
                uint2 rw[NLD];
#pragma unroll
                for (int i = 0; i < NLD; ++i) {
                    const int q = gt + i * NCONV;
                    rw[i] = q < NPAIR ? reinterpret_cast<const uint2 *>(rawt)[q] : make_uint2(0u, 0u);
                }
#pragma unroll
                for (int i = 0; i < NLD; ++i) {
                    const float2 s0 = widen_iq16(rw[i].x, a.in_scale), s1 = widen_iq16(rw[i].y, a.in_scale);
                    raw[i] = make_float4(s0.x, s0.y, s1.x, s1.y);
                }
                if (t0 < HALO || t0 + TILE > ((long long)a.n & ~3ll)) {
#pragma unroll
                    for (int i = 0; i < NLD; ++i) {
                        const int q = gt + i * NCONV;
                        const long long g = t0 - HALO + 2 * q;  // even
                        if (q < NPAIR && (g < 0 || g + 1 >= ((long long)a.n & ~3ll))) raw[i] = iq16_edge_pair(a, g, HALO);
                    }
                    if (t0 < HALO) {
#pragma unroll
                        for (int i = 0; i < NLD; ++i) {
                            const float4 v = raw[i];
                            mnu = min(mnu, quiet_key<SMIN>(v, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)))));
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < NLD; ++i) {
                    const float4 v = raw[i];
                    mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
                }
            } else {
#pragma unroll
                for (int i = 0; i < NLD; ++i) {
                    const int q = gt + i * NCONV;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (q < NPAIR) {
                        const long long g = t0 - HALO + 2 * q;  // even
                        if (g < 0 || g + 1 < (long long)a.n) {
                            v = rawt[q];
                        } else if (g < (long long)a.n) {  // odd trailing sample: not covered by the 16-byte bulk copies
                            const float2 t = a.x[g];
                            v = make_float4(t.x, t.y, 0.f, 0.f);
                        }
                    }
                    raw[i] = v;
                    const float pm = fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));
                    mx = fmaxf(mx, pm);
                    mnu = min(mnu, quiet_key<SMIN>(v, pm));
                }
            }
            mbar_arrive(&raw_empty[rs]);  // tile is in registers: the TMA warp may refill the stage
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                mnu = min(mnu, __shfl_xor_sync(0xffffffffu, mnu, o));
            }
            if (lane == 0) {
                red_max[s][ph][gw] = mx;
                red_min[s][ph][gw] = mnu;
            }
            FTC_T(gt == 0, 2);
            asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "n"(NCONV) : "memory");
            FTC_T(gt == 0, 3);
            mx = red_max[s][ph][0];
            mnu = red_min[s][ph][0];
#pragma unroll
            for (int w = 1; w < NCW; ++w) {
                mx = fmaxf(mx, red_max[s][ph][w]);
                mnu = min(mnu, red_min[s][ph][w]);
            }
            // a quiet stretch more than 2^20 below the tile maximum (its lo terms go denormal): this tile is recomputed
            // in plain f32 by the fix-up pass (FirFix); non-finite samples are caught in the conversion loop below
            if (gt == 0 && a.fix_count != nullptr && mnu != 0xffffffffu && __uint_as_float(mnu + 1u) < mx * 9.5367431640625e-7f &&
                atomicExch(&fix_seen[s], (unsigned)tile + 1u) != (unsigned)tile + 1u)
                a.fix_list[atomicAdd(a.fix_count, 1u)] = (unsigned)tile;
            // exact power-of-two block scale: max * sc in [2^14, 2^15)
            uint32_t eb = (__float_as_uint(mx) >> 23) & 0xFF;
            eb = (eb < 16 || eb == 255) ? 141 : eb;  // all-zero / denormal / non-finite tile: scale 1
            const float sc = __uint_as_float((268u - eb) << 23);
            if (gt == 0) {  // the epilogue is at most 4 tiles behind: an 8-deep ring cannot wrap
                inv_scale[it & 7] = __uint_as_float((eb - 14u) << 23);
                mbar_arrive(&sc_ready[it & 7]);
            }

            FTC_T(gt == 0, 4);
            mbar_wait(&a_empty[s], ph ^ 1);  // MMAs that read this stage two tiles ago are done
            FTC_T(gt == 0, 5);
            unsigned char *hi = sA + s * A_STAGE, *lo = hi + A_PART;
            __half2 nanacc = __floats2half2_rn(0.f, 0.f);  // sum of the lo terms: NaN iff a sample of the tile is Inf / NaN
#pragma unroll
            for (int i = 0; i < NLD; ++i) {
                const int q = gt + i * NCONV;
                if (q < NPAIR) {
                    const float4 v = make_float4(raw[i].x * sc, raw[i].y * sc, raw[i].z * sc, raw[i].w * sc);
                    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
                    const float2 b0 = __half22float2(h0), b1 = __half22float2(h1);
                    const __half2 l0 = __floats2half2_rn(v.x - b0.x, v.y - b0.y);
                    const __half2 l1 = __floats2half2_rn(v.z - b1.x, v.w - b1.y);
                    nanacc = __hadd2(nanacc, __hadd2(l0, l1));  // Inf * sc - Inf = NaN, NaN stays NaN; finite |lo| < 16
                    const uint32_t off = swz128((uint32_t)q * 8u);
                    uint2 ph2, pl2;
                    ph2.x = *reinterpret_cast<const uint32_t *>(&h0);
                    ph2.y = *reinterpret_cast<const uint32_t *>(&h1);
                    pl2.x = *reinterpret_cast<const uint32_t *>(&l0);
                    pl2.y = *reinterpret_cast<const uint32_t *>(&l1);
                    *reinterpret_cast<uint2 *>(hi + off) = ph2;
                    *reinterpret_cast<uint2 *>(lo + off) = pl2;
                }
            }
            fence_proxy_async();
            mbar_arrive(&a_full[s]);
            FTC_T(gt == 0, 6);
            if (a.fix_count != nullptr && (__hisnan(__low2half(nanacc)) || __hisnan(__high2half(nanacc))) &&
                atomicExch(&fix_seen[s], (unsigned)tile + 1u) != (unsigned)tile + 1u)
                a.fix_list[atomicAdd(a.fix_count, 1u)] = (unsigned)tile;  // non-finite sample: exact fall-back (FirFix)
        }
        FTC_OUT(gt == 0, 1 + grp);
    } else if (warp == W_MMA) {
        // ------------------------------------------------------------------ MMA issuer
        // The whole warp runs the loop, one elected lane issues: inside `if (lane == 0)` the compiler cannot prove the
        // descriptors warp-uniform and wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST / branch sequence (~14
        // instructions per MMA on a scheduler shared with busy warps); warp-uniform code keeps them in uniform registers
        // (descriptor = base descriptor + (byte offset >> 4), one UIADD3.64 between two UTCHMMAs).
        unsigned long long it = 0;
        const uint64_t bd0 = tc_desc(smem_u32(sB)), ad0 = tc_desc(smem_u32(sA));
        FTC_DECL;
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = (int)(it & 1);
            const uint32_t ph = (uint32_t)((it >> 1) & 1);
            FTC_T(lane == 0, 0);
            mbar_wait_long(&t_empty[s], ph ^ 1);
            FTC_T(lane == 0, 1);
            mbar_wait_long(&a_full[s], ph);
            FTC_T(lane == 0, 2);
            tc_fence_after();
            const uint64_t ahi = ad0 + (uint64_t)((s * A_STAGE) >> 4), alo = ahi + (uint64_t)(A_PART >> 4);
            const uint32_t d = tmem_base + (uint32_t)s * 128u;
            if (elect_one()) {
#pragma unroll
                for (int t = 0; t < KB * 4; ++t) {
                    const uint64_t aoff = (uint64_t)(((t >> 2) * 128 + (t & 3) * 32) >> 4);
                    const uint64_t boff = (uint64_t)(((t >> 2) * 16384 + (t & 3) * 32) >> 4);
                    tc_mma(d, ahi + aoff, bd0 + boff, IDESC128, t > 0 ? 1u : 0u);
                    tc_mma(d, alo + aoff, bd0 + boff, IDESC64, 1u);
                }
                tc_commit(&a_empty[s]);
                tc_commit(&t_full[s]);
            }
            __syncwarp();
        }
        FTC_OUT(lane == 0, 3);
    } else {
        // ------------------------------------------------------------------ epilogue
        const int e = warp - W_EPI;  // TMEM sub-partition = warp % 4
        unsigned char *stage = sOut + e * OUT_WARP;
        const bool direct = IQ16 ? (reinterpret_cast<uintptr_t>(a.y16) & 31) == 0 : (reinterpret_cast<uintptr_t>(a.y) & 31) == 0;
        unsigned long long it = 0;
        FTC_DECL;
        for (unsigned long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int s = (int)(it & 1);
            const uint32_t ph = (uint32_t)((it >> 1) & 1);
            const long long t0 = (long long)tile * TILE;
            FTC_T(e == 0 && lane == 0, 0);
            mbar_wait(&sc_ready[it & 7], (uint32_t)((it >> 3) & 1));  // acquire the loaders' block scale
            const float k0 = inv_scale[it & 7], k1 = a.tap_inv_scale;
            mbar_wait_long(&t_full[s], ph);
            FTC_T(e == 0 && lane == 0, 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * e) << 16) + (uint32_t)s * 128u;
            // Lane m of this warp owns row 32 e + m of the tile = 32 consecutive output samples (256 bytes).  With the
            // y pointer 32-byte aligned the row goes out as 8 x 256-bit stores (whole sectors, no shared-memory
            // transpose: the staging round trip was 16 B/sample of shared-memory traffic on the busiest pipe);
            // otherwise through the padded per-warp staging buffer and 128-bit coalesced stores.
            const long long row = t0 + (long long)(32 * e + lane) * RS;
            if constexpr (IQ16) {
                // 32 output samples = 128 bytes of i16 IQ per lane: 4 x 256-bit stores of 8 words (whole sectors) when
                // y16 is 32-byte aligned, single words otherwise.  (out_scale * y) as i16 with y formed exactly as the
                // f32 epilogue forms it, so the words equal quantising the f32 result.
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t p[32], r[32];
                    tc_ld32(taddr + half * 32, p);
                    tc_ld32(taddr + 64 + half * 32, r);
                    tc_wait_ld();
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        float w[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const float vr = (__uint_as_float(p[16 * c + 2 * u]) + __uint_as_float(r[16 * c + 2 * u])) * k0 * k1;
                            const float vi = (__uint_as_float(p[16 * c + 2 * u + 1]) + __uint_as_float(r[16 * c + 2 * u + 1])) * k0 * k1;
                            w[u] = __uint_as_float(pack_i16(quant_i16(vr, a.out_scale), quant_i16(vi, a.out_scale)));
                        }
                        const long long sidx = row + 16 * half + 8 * c;  // 8 complex samples = 32 bytes
                        if (direct && sidx + 7 < (long long)a.n) {
                            stg_stream8(reinterpret_cast<float *>(a.y16 + sidx), w);
                        } else {
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (sidx + u < (long long)a.n) a.y16[sidx + u] = __float_as_uint(w[u]);
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(&t_empty[s]);
                FTC_T(e == 0 && lane == 0, 2);
                continue;
            }
            if (direct) {
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    uint32_t p[32], r[32];
                    tc_ld32(taddr + half * 32, p);
                    tc_ld32(taddr + 64 + half * 32, r);
                    tc_wait_ld();
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float v[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u)
                            v[u] = (__uint_as_float(p[8 * c + u]) + __uint_as_float(r[8 * c + u])) * k0 * k1;
                        const long long sidx = row + 16 * half + 4 * c;  // 4 complex samples = 32 bytes
                        if (sidx + 3 < (long long)a.n) {
                            stg_stream8(reinterpret_cast<float *>(a.y + sidx), v);
                        } else {
#pragma unroll
                            for (int u = 0; u < 4; ++u)
                                if (sidx + u < (long long)a.n) a.y[sidx + u] = make_float2(v[2 * u], v[2 * u + 1]);
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(&t_empty[s]);
                FTC_T(e == 0 && lane == 0, 2);
                continue;
            }
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                uint32_t p[32], r[32];
                tc_ld32(taddr + half * 32, p);
                tc_ld32(taddr + 64 + half * 32, r);
                tc_wait_ld();
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float4 v;
                    v.x = (__uint_as_float(p[4 * c]) + __uint_as_float(r[4 * c])) * k0 * k1;
                    v.y = (__uint_as_float(p[4 * c + 1]) + __uint_as_float(r[4 * c + 1])) * k0 * k1;
                    v.z = (__uint_as_float(p[4 * c + 2]) + __uint_as_float(r[4 * c + 2])) * k0 * k1;
                    v.w = (__uint_as_float(p[4 * c + 3]) + __uint_as_float(r[4 * c + 3])) * k0 * k1;
                    *reinterpret_cast<float4 *>(stage + lane * OUT_PITCH + half * 128 + c * 16) = v;
                }
            }
            tc_fence_before();
            mbar_arrive(&t_empty[s]);
            __syncwarp();
            // 32 rows x 256 B of this warp = 8 KB contiguous in y
            const long long row0 = t0 + (long long)(32 * e) * RS;
#pragma unroll 4
            for (int i = 0; i < 16; ++i) {
                const int idx = i * 32 + lane, rr = idx >> 4, c = idx & 15;
                const float4 v = *reinterpret_cast<const float4 *>(stage + rr * OUT_PITCH + c * 16);
                const long long sidx = row0 + (long long)rr * RS + 2 * c;
                if (sidx + 1 < (long long)a.n) stg_stream(reinterpret_cast<float4 *>(a.y + sidx), v);
                else if (sidx < (long long)a.n) a.y[sidx] = make_float2(v.x, v.y);
            }
            __syncwarp();
            FTC_T(e == 0 && lane == 0, 2);
        }
        FTC_OUT(e == 0 && lane == 0, 4);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == W_MMA) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256) : "memory");
    }
}

// samples g, g + 1 of the stream seen by an IQ16 tile where they are not in its raw words: before the batch (f32 history)
// or in the unaligned tail (read from the i16 words directly), zero past the end
__device__ __noinline__ float4 iq16_edge_pair(const Args &a, long long g, int halo)
{
    float2 s0 = make_float2(0.f, 0.f), s1 = s0;
    if (g < 0) {
        s0 = a.halo[halo + g];
        s1 = a.halo[halo + g + 1];
    } else {
        if (g < (long long)a.n) s0 = widen_iq16(a.x16[g], a.in_scale);
        if (g + 1 < (long long)a.n) s1 = widen_iq16(a.x16[g + 1], a.in_scale);
    }
    return make_float4(s0.x, s0.y, s1.x, s1.y);
}

}  // namespace tc

// ------------------------------------------------------------------------------------ host side
// B image for KB K-blocks: region kb (16 KiB) = 128 rows x 128 bytes, row n < 64: fp16 hi part of
// B[n][64 kb .. 64 kb + 63], row 64 + n: the lo part; 128-byte swizzled like the device reads it.
size_t fir_tc_image_bytes(uint32_t ntaps)
{
    const int kb = 1 + (int)ceil_div(ntaps ? ntaps : 1, (size_t)tc::RS);
    return (size_t)kb * 16384;
}

int fir_tc_kblocks(uint32_t ntaps) { return 1 + (int)ceil_div(ntaps ? ntaps : 1, (size_t)tc::RS); }

void fir_tc_build_image(const float2 *taps, uint32_t ntaps, unsigned char *img, float *tap_inv_scale)
{
    const int KB = fir_tc_kblocks(ntaps);
    const int HALO = tc::RS * (KB - 1);
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
    memset(img, 0, (size_t)KB * 16384);
    for (int n = 0; n < 64; ++n) {
        const int i = n >> 1, c = n & 1;
        for (int k = 0; k < 64 * KB; ++k) {
            const int j = k >> 1, d = k & 1;
            const int t = i + HALO - j;
            float v = 0.f;
            if (t >= 0 && t < (int)ntaps) {
                const float hr = taps[t].x, hi = taps[t].y;
                v = c == 0 ? (d == 0 ? hr : -hi) : (d == 0 ? hi : hr);
            }
            v *= sc;
            const __half h = __float2half_rn(v);
            const __half l = __float2half_rn(v - __half2float(h));
            const int kb = k >> 6, kk = k & 63;
            uint32_t o_hi = (uint32_t)n * 128u + (uint32_t)kk * 2u;
            uint32_t o_lo = (uint32_t)(64 + n) * 128u + (uint32_t)kk * 2u;
            o_hi ^= ((o_hi >> 7) & 7) << 4;
            o_lo ^= ((o_lo >> 7) & 7) << 4;
            memcpy(img + (size_t)kb * 16384 + o_hi, &h, 2);
            memcpy(img + (size_t)kb * 16384 + o_lo, &l, 2);
        }
    }
}

template <int KB, bool IQ16, bool SMIN>
static int launch_tc_kb(const tc::Args &a, cudaStream_t stream)
{
    constexpr int RAWB = (tc::TILE + tc::RS * (KB - 1)) * (IQ16 ? 4 : 8);
    constexpr int BASE = KB * 16384 + 2 * tc::A_STAGE + 4 * tc::OUT_WARP + 1024;
    constexpr int NRAW = BASE + 2 * RAWB <= 227 * 1024 ? 2 : 1;
    constexpr int SMEM = BASE + NRAW * RAWB;
    static_assert(SMEM <= 227 * 1024, "fir_tc: shared memory budget");
    auto kern = tc::fir_tc_kernel<KB, NRAW, IQ16, SMIN>;
    CB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    const unsigned long long ntiles = (a.n + tc::TILE - 1) / tc::TILE;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned grid = (unsigned)(ntiles < (unsigned long long)sms ? ntiles : (unsigned long long)sms);
    kern<<<grid, tc::NTHREADS, SMEM, stream>>>(a);
    count_launch();
    CB_CUDA(cudaGetLastError());
    return CB_OK;
}

bool fir_tc_applicable(const FirSeg &seg)
{
    if (seg.interp != 1 || seg.decim != 1 || seg.ntaps == 0 || seg.ntaps > 128) return false;
    const int KB = fir_tc_kblocks(seg.ntaps);
    const uint32_t halo = (uint32_t)tc::RS * (KB - 1);
    if (seg.hist_len < halo) return false;
    const float2 *h = seg.hist_in + (seg.hist_len - halo);
    return ((reinterpret_cast<uintptr_t>(seg.x) | reinterpret_cast<uintptr_t>(seg.y) | reinterpret_cast<uintptr_t>(h)) & 15) == 0;
}

// i16 IQ on both edges: applicable like the f32 form, on 16-byte aligned word buffers
bool fir_tc_iq16_applicable(const FirSeg &seg, const int16_t *x16, const int16_t *y16)
{
    if (seg.interp != 1 || seg.decim != 1 || seg.ntaps == 0 || seg.ntaps > 128) return false;
    const int KB = fir_tc_kblocks(seg.ntaps);
    const uint32_t halo = (uint32_t)tc::RS * (KB - 1);
    if (seg.hist_len < halo) return false;
    return (reinterpret_cast<uintptr_t>(x16) & 15) == 0 && (reinterpret_cast<uintptr_t>(y16) & 3) == 0;
}

// the kernel for the plan's tap count and quiet test, then the exact fall-back pass over the tiles it flagged
static int launch_tc(const FirSeg &seg, tc::Args &a, bool iq16, const FirTcPlan &plan, const float2 *taps_dev,
                     cudaStream_t stream)
{
    if (seg.n_in == 0) return CB_OK;
    const int KB = fir_tc_kblocks(seg.ntaps);
    a.halo = seg.hist_in + (seg.hist_len - (uint32_t)tc::RS * (KB - 1));
    a.hist_in = seg.hist_in;
    a.hist_out = seg.hist_out;
    a.bimg = reinterpret_cast<const uint4 *>(plan.bimg_dev);
    a.n = seg.n_in;
    a.hist_len = seg.hist_len;
    a.tap_inv_scale = plan.tap_inv_scale;
    FirFix *fix = plan.fix;
    const bool fixup = fix != nullptr && fix->dev != nullptr && taps_dev != nullptr &&
                       fix->cap >= ceil_div(seg.n_in, (size_t)tc::TILE);
    a.fix_count = fixup ? fix->dev + (fix->calls & 1u) : nullptr;
    a.fix_list = fixup ? fix->dev + 2 : nullptr;
    const int sel = KB * 4 + (iq16 ? 2 : 0) + (plan.sample_min ? 1 : 0);
    int rc;
    switch (sel) {
#define CB_TC_CASE(kb)                                                          \
    case kb * 4 + 0: rc = launch_tc_kb<kb, false, false>(a, stream); break; \
    case kb * 4 + 1: rc = launch_tc_kb<kb, false, true>(a, stream); break;  \
    case kb * 4 + 2: rc = launch_tc_kb<kb, true, false>(a, stream); break;  \
    case kb * 4 + 3: rc = launch_tc_kb<kb, true, true>(a, stream); break;
    CB_TC_CASE(2)
    CB_TC_CASE(3)
    CB_TC_CASE(4)
    CB_TC_CASE(5)
#undef CB_TC_CASE
    default: set_error("fir_tc: unsupported tap count %u", seg.ntaps); return CB_ERR_UNSUPPORTED;
    }
    if (rc || !fixup) return rc;
    FirFixArgs f{a.x, seg.hist_in, taps_dev, a.y, reinterpret_cast<int16_t *>(a.y16), a.out_scale, seg.n_in, seg.ntaps, 1u,
                 (unsigned)tc::TILE, seg.hist_len, a.fix_count, fix->dev + ((fix->calls + 1) & 1u), a.fix_list, a.x16, a.in_scale};
    ++fix->calls;
    return launch_fir_fixup(f, stream);
}

int launch_fir_tc_iq16(const FirSeg &seg, const int16_t *x16, float in_scale, int16_t *y16, float out_scale,
                       const FirTcPlan &plan, const float2 *taps_dev, cudaStream_t stream)
{
    tc::Args a = {};
    a.x16 = reinterpret_cast<const uint32_t *>(x16);
    a.y16 = reinterpret_cast<uint32_t *>(y16);
    a.in_scale = in_scale;
    a.out_scale = out_scale;
    return launch_tc(seg, a, true, plan, taps_dev, stream);
}

int launch_fir_tc(const FirSeg &seg, const FirTcPlan &plan, const float2 *taps_dev, cudaStream_t stream)
{
    tc::Args a = {};
    a.x = seg.x;
    a.y = seg.y;
    a.out_scale = 1.f;
    return launch_tc(seg, a, false, plan, taps_dev, stream);
}

}  // namespace cb
