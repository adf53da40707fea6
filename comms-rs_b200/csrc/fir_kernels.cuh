// FIR kernels (K1 / K3 of SURVEY.md section 2): device code + launch wrappers.
//
// Reference semantics (src/filter/fir.rs:87-102):
//   y[n] = sum_{k<K} h[k] * x[n-k],   x[-1-k] = state[k]
// The K-1 samples before a batch (the reference's `state`) are exactly an
// overlap-save halo, so every tile of outputs is independent given its input
// range plus a K-sample halo.
#pragma once
#include "common.cuh"

namespace cb {

// One launch of a FIR over a contiguous segment.
struct FirSeg {
    const float2 *x;        // n_in input samples (device)
    const float2 *hist_in;  // hist_len samples preceding x[0], chronological (oldest first)
    float2 *hist_out;       // may be NULL; receives the last hist_len samples of [hist_in ++ x]
    float2 *y;              // outputs
    size_t n_in;
    size_t n_out;
    uint32_t hist_len;      // >= taps-per-phase halo, even
    uint32_t ntaps;         // effective taps (min(len taps, len state)), > 0
    uint32_t interp;        // L >= 1
    uint32_t decim;         // D >= 1
    int16_t *y16 = nullptr; // fused quantiser: write (qscale * y) as interleaved i16 IQ here instead of y
    float qscale = 1.f;     //   (only the polyphase tensor-core kernel fuses it; see launch_fir_i16)
};

// Work list of the tensor-core kernels' exact fall-back.  The tensor-core filters scale a whole tile by one power of
// two before the two-term fp16 split, which holds f32-level accuracy only while a tile's quiet stretches stay within
// ~2^-20 of its maximum, and a single Inf / NaN poisons every product of the tile.  The converter warps therefore
// flag such tiles (non-finite sample, or a pair of adjacent samples below 2^-20 of the tile maximum -- each sample on its
// own for filters with parity-sparse taps, FirTcPlan::sample_min) and append them here; fir_fixup_kernel, launched behind every tensor-core launch, recomputes exactly those tiles in plain f32 direct
// form (the reference's arithmetic, src/filter/fir.rs:87-102) and overwrites them.  dev[0], dev[1]: counters used by
// alternate launches (the fix-up kernel of launch k zeroes the counter of launch k+1); dev[2..]: tile indices.
struct FirFix {
    unsigned *dev = nullptr;
    unsigned cap = 0;       // tile indices the list can hold
    unsigned calls = 0;     // launches so far (selects the counter)
};

// Tensor-core path (fir_tc_kernel.cu): prepacked fp16 hi/lo Toeplitz tap image + its scale.
struct FirTcPlan {
    const void *bimg_dev;   // fir_tc_image_bytes(ntaps) bytes, device
    float tap_inv_scale;
    size_t min_samples;     // use the tensor-core kernel from this batch size on
    FirFix *fix = nullptr;  // the launch's fix-up list (one per concurrent lane); NULL: no fall-back pass
    bool sample_min = false;  // quiet test per sample instead of per 16-byte pair (fir_taps_pair_sparse)
};
// The quiet test looks at 16-byte pairs of complex samples (x[2j], x[2j+1]): it sees every output formed from quiet
// samples only if the taps always reach both samples of some pair, i.e. if the (per phase) taps hold two adjacent
// non-zero entries ending at an even offset and two ending at an odd one.  Taps without (one tap, every other tap
// zero, two taps) need the per-sample test; the dense filters keep the cheaper pair test.
bool fir_taps_pair_sparse(const float2 *taps, uint32_t ntaps, uint32_t interp);

// Key of that test for a 16-byte pair (re0, im0, re1, im1) with pair maximum pm: the smallest non-zero magnitude
// minus one (a zero wraps to the top) -- of the pair, or with SMIN of each sample
template <bool SMIN>
__device__ __forceinline__ uint32_t quiet_key(float4 v, float pm)
{
    if constexpr (SMIN)
        return min(__float_as_uint(fmaxf(fabsf(v.x), fabsf(v.y))) - 1u, __float_as_uint(fmaxf(fabsf(v.z), fabsf(v.w))) - 1u);
    else
        return __float_as_uint(pm) - 1u;
}
// upper bound of the tiles any tensor-core launch over n_in inputs can flag
static inline size_t fir_fix_tiles(size_t n_in) { return n_in / 512 + 8; }

struct FirFixArgs {
    const float2 *x, *hist_in, *taps;
    float2 *y;
    int16_t *y16;
    float qscale;
    unsigned long long n;   // input samples
    unsigned ntaps, interp, tile_in, hist_len;
    const unsigned *count;
    unsigned *next_count;
    const unsigned *list;
    const uint32_t *x16 = nullptr;  // i16 IQ input words instead of x (x = in_scale * (i16 as f32), like cb_convert_i16)
    float in_scale = 1.f;
};
int launch_fir_fixup(const FirFixArgs &a, cudaStream_t stream);
size_t fir_tc_image_bytes(uint32_t ntaps);
int fir_tc_kblocks(uint32_t ntaps);
void fir_tc_build_image(const float2 *taps, uint32_t ntaps, unsigned char *img, float *tap_inv_scale);
bool fir_tc_applicable(const FirSeg &seg);
int launch_fir_tc(const FirSeg &seg, const FirTcPlan &plan, const float2 *taps_dev, cudaStream_t stream);
bool fir_tc_iq16_applicable(const FirSeg &seg, const int16_t *x16, const int16_t *y16);
// with the same exact fall-back as launch_fir_tc (the first tile's halo is the f32 history, which can hold anything)
int launch_fir_tc_iq16(const FirSeg &seg, const int16_t *x16, float in_scale, int16_t *y16, float out_scale,
                       const FirTcPlan &plan, const float2 *taps_dev, cudaStream_t stream);

// Polyphase tensor-core path (fir_ptc_kernel.cu): interp in {4, 8}, decim = 1, real or complex taps.
// The plan's bimg_dev / tap_inv_scale then hold the polyphase tap image.
bool fir_ptc_supported(uint32_t ntaps, uint32_t interp, bool taps_real);
int fir_ptc_ksteps(uint32_t ntaps, uint32_t interp);
size_t fir_ptc_image_bytes(uint32_t ntaps, uint32_t interp, bool taps_real);
void fir_ptc_build_image(const float2 *taps, uint32_t ntaps, uint32_t interp, bool taps_real, unsigned char *img,
                         float *tap_inv_scale);
bool fir_ptc_applicable(const FirSeg &seg, bool taps_real);
int launch_fir_ptc(const FirSeg &seg, const FirTcPlan &plan, bool taps_real, const float2 *taps_dev, cudaStream_t stream);

// Overlap-save path for long filters (fft_kernels.cu): 129 .. 1025 taps, decim = interp = 1.
// hf: 4096-point spectrum of the zero-padded taps; tw_fwd / tw_inv: fft2 tables for 4096 points; spec: scratch of
// fir_ols_frames(n, ntaps) * 4096 complex samples.
size_t fir_ols_frames(size_t n, uint32_t ntaps);
int launch_fir_ols(const float2 *x, size_t n, const float2 *hist_in, float2 *hist_out, uint32_t hist_len, uint32_t ntaps,
                   const float2 *hf, const float2 *tw_fwd, const float2 *tw_inv, float2 *spec, float2 *y, cudaStream_t s);

// Real-input / real-output decimating FIR (fir_real_kernel.cu): x -> Complex(x, 0) -> FIR -> .re -> every D-th, fused.
// interp = 1, <= 64 taps, D in {2, 4, 5, 8, 10}; hist_in / hist_out are the handle's complex history buffers.
bool fir_real_applicable(uint32_t ntaps, uint32_t interp, uint32_t decim);
int launch_fir_real(const float *x, size_t n_in, const float2 *hist_in, float2 *hist_out, uint32_t hist_len,
                    const float2 *taps_host, uint32_t ntaps, uint32_t decim, float *y, cudaStream_t s);

// taps_dev: ntaps complex taps in device memory (generic path)
// taps_host: same on the host (fast paths put them in the kernel parameter constant bank)
// tcplan: NULL = CUDA-core kernels only
int launch_fir(const FirSeg &seg, const float2 *taps_dev, const float2 *taps_host, bool taps_real,
               const FirTcPlan *tcplan, cudaStream_t stream);
// true when launch_fir would take a kernel that writes seg.y16 itself (otherwise the caller filters into
// an f32 scratch and runs the stand-alone quantiser)
bool fir_fuses_i16(const FirSeg &seg, bool taps_real, const FirTcPlan *tcplan);

}  // namespace cb
