// Complex<f64> FFT (cb_fft_f64): launch wrappers of the kernels in fft_f64_kernels.cu.  The arithmetic they share with
// the CPU emulation is in fft64_core.cuh.
#pragma once
#include "common.cuh"

namespace cb {

// Transforms of n = 2^log2n points (8 <= n <= 4096), one per column: `frames` frames of `cols` columns each; element
// j of column c of frame f is in[f in_f + c in_c + j in_j], output bin k goes to out[f out_f + c out_c + k out_k].
// tw holds e^{-/+ 2 pi i e / (tw_step n)}.  With twist non-NULL, output k of column c is multiplied by twist[k c]
// before the store (the inter-step twiddle of a two-step transform).
struct Fft64Cols {
    const double2 *in;
    double2 *out;
    const double2 *tw;
    const double2 *twist;
    size_t in_j, in_c, in_f, out_k, out_c, out_f;
    unsigned tw_step, log2n, cols;
    size_t frames;
};
int launch_fft64_cols(const Fft64Cols &a, int inverse, cudaStream_t s);

// Direct sums X[k] = sum_n x[n] tw[kn mod n] over frames of n points (tw: the n-entry table of the plan's sign).
int launch_fft64_direct(const double2 *in, double2 *out, const double2 *tw, unsigned n, size_t frames, cudaStream_t s);

// Chirp-z steps over frames of n points padded to m: a = x chirp (zero past n); spec *= bspec; out = c chirp.
int launch_fft64_chirp_pre(const double2 *x, const double2 *chirp, double2 *a, unsigned n, unsigned m, size_t frames,
                           cudaStream_t s);
int launch_fft64_chirp_mul(double2 *spec, const double2 *bspec, unsigned m, size_t frames, cudaStream_t s);
int launch_fft64_chirp_post(const double2 *c, const double2 *chirp, double2 *out, unsigned n, unsigned m, size_t frames,
                            cudaStream_t s);

}  // namespace cb
