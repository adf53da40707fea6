// Complex<f64> FIR (batch_fir over Complex<f64>, src/filter/fir.rs:87-102): device code + launch wrapper.
//
// Every output is two FMA chains (real part, imaginary part) that start from +0 and run over the output's taps in
// ascending tap index, and only over taps that meet a real input sample (never a stuffed zero, a padding tap or history
// older than the state).  The order depends on nothing else -- not the tile, the tap chunk, the call split, decim or
// the kernel -- so every kernel below produces the same bits for the same output.
#pragma once
#include "common.cuh"

namespace cb {

// One launch of the f64 FIR over a contiguous segment (the f64 twin of FirSeg).
struct Fir64Seg {
    const double2 *x;        // n_in input samples (device, 16-byte aligned)
    const double2 *hist_in;  // hist_len samples preceding x[0], chronological (oldest first)
    double2 *hist_out;       // may be NULL; receives the last hist_len samples of [hist_in ++ x]
    double2 *y;              // n_out outputs
    size_t n_in;
    size_t n_out;
    uint32_t hist_len;       // >= the taps' reach into the past, in input samples
    uint32_t ntaps;          // effective taps, min(len taps, len state)
    uint32_t interp;         // L >= 1
    uint32_t decim;          // D >= 1
};

// taps_dev: ntaps complex taps (device).  taps_real: every imaginary part is zero (2 instead of 4 FMAs per term).
int launch_fir_f64(const Fir64Seg &seg, const double2 *taps_dev, bool taps_real, cudaStream_t stream);

}  // namespace cb
