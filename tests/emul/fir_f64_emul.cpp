// CPU emulation of the Complex<f64> FIR's numerical contract (include/comms_b200.h, cb_fir_f64): every output is two
// FMA chains from +0 over the output's taps in ascending tap index, only over taps that meet a real input sample.
// Built as a shared library (g++ -O2 -ffp-contract=off -fopenmp -shared -fPIC ... -lquadmath) and called through
// ctypes by tests/test_fir_f64_cpu.py and tests/test_gpu_fir_f64.py.
//
// Beside the device bits it returns, per output: the exact value (a __float128 sum of the exact products, as a
// double-double), |y - exact| (complex modulus), A_n = sum |h_k| |x_{n-k}| over the chain's taps, K_n (the chain's
// length) and whether the chain reaches a non-finite sample.  `mutation` != 0 reproduces one defect the tests must
// reject (see the enum).
#include <quadmath.h>

#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

namespace {

enum Mutation {
    NONE = 0,
    HALO_SEAM = 1,     // outputs at a 2048-output tile seam miss the term of tap 1 (a halo sample)
    DROP_LAST = 2,     // every chain drops its last tap
    ZERO_HIST = 3,     // the second call starts from a zero history
    PAD_TAP = 4,       // the chain runs over taps padded with zeros to a multiple of 8 (0 * Inf = NaN)
    DECIM_CARRY = 5,   // the decimation phase carries over calls instead of resetting
};

}  // namespace

extern "C" long fir64_emul(const double *taps, size_t ntaps, const double *state, size_t nstate, int has_state,
                           unsigned decim, unsigned interp, const double *x, const size_t *calls, size_t ncalls,
                           int mutation, int want_exact, double *y, double *exact_hi, double *exact_lo, double *err,
                           double *amag, uint32_t *kn, uint8_t *reach_bad, size_t cap)
{
    const size_t D = decim ? decim : 1, L = interp ? interp : 1;
    const size_t ns = has_state ? nstate : ntaps;
    const size_t K = ntaps < ns ? ntaps : ns;
    // the stream: input-domain history (the state's on-grid entries, oldest first) followed by every input sample
    const size_t H = ((ns > K ? ns : K) + L - 1) / L;
    std::vector<double> s(2 * H, 0.0);
    if (has_state) {
        for (size_t k = 0; k < nstate; ++k) {
            const double re = state[2 * k], im = state[2 * k + 1];
            if ((k + 1) % L == 0) {
                const size_t i = (k + 1) / L;
                if (i <= H) {
                    s[2 * (H - i)] = re;
                    s[2 * (H - i) + 1] = im;
                }
            } else if (re != 0.0 || im != 0.0) {
                return -1;  // CB_ERR_UNSUPPORTED
            }
        }
    }
    size_t total = 0;
    for (size_t c = 0; c < ncalls; ++c) total += calls[c];
    s.insert(s.end(), x, x + 2 * total);
    bool cplx = false;
    for (size_t k = 0; k < K; ++k) cplx |= taps[2 * k + 1] != 0.0;
    const size_t Kpad = mutation == PAD_TAP ? (K + 7) / 8 * 8 : K;

    // (call, first input, first output, stuffed-domain offset of the first surviving output) for each call
    struct Call { size_t in0, m, out0, u0, nout; };
    std::vector<Call> cl;
    size_t in0 = 0, out0 = 0, stuffed = 0;
    for (size_t c = 0; c < ncalls; ++c) {
        const size_t m = calls[c], up = m * L;
        size_t u0 = 0;
        if (mutation == DECIM_CARRY) u0 = (D - stuffed % D) % D;
        const size_t nout = up > u0 ? (up - u0 + D - 1) / D : 0;
        cl.push_back({in0, m, out0, u0, nout});
        in0 += m;
        out0 += nout;
        stuffed += up;
    }
    if (out0 > cap) return -2;

    for (size_t c = 0; c < cl.size(); ++c) {
        const Call C = cl[c];
#pragma omp parallel for schedule(static)
        for (long long qq = 0; qq < (long long)C.nout; ++qq) {
            const size_t q = (size_t)qq;
            const size_t u = C.u0 + q * D, p = u % L;
            const long long mm = (long long)(u / L);
            double re = 0.0, im = 0.0;
            __float128 er = 0, ei = 0, a = 0;
            uint32_t cnt = 0;
            bool bad = false;
            long long idx = mm;  // input index within the call; the stream position is H + in0 + idx
            for (size_t k = p; k < Kpad; k += L, --idx) {
                const long long pos = (long long)H + (long long)C.in0 + idx;
                if (pos < 0) break;  // older than the state: no term
                double xr = s[2 * pos], xi = s[2 * pos + 1];
                if (mutation == ZERO_HIST && c == 1 && idx < 0) xr = xi = 0.0;
                if (mutation == DROP_LAST && k + L >= K) break;
                if (mutation == HALO_SEAM && k == 1 && (C.out0 + q) % 2048 == 0 && C.out0 + q > 0) continue;
                const double hr = k < K ? taps[2 * k] : 0.0, hi = k < K ? taps[2 * k + 1] : 0.0;
                re = std::fma(hr, xr, re);
                if (cplx) re = std::fma(-hi, xi, re);
                im = std::fma(hr, xi, im);
                if (cplx) im = std::fma(hi, xr, im);
                ++cnt;
                bad |= !std::isfinite(xr) || !std::isfinite(xi);
                if (want_exact) {
                    er += (__float128)hr * xr - (__float128)hi * xi;
                    ei += (__float128)hr * xi + (__float128)hi * xr;
                    a += (__float128)std::hypot(hr, hi) * (__float128)std::hypot(xr, xi);
                }
            }
            const size_t o = C.out0 + q;
            y[2 * o] = re;
            y[2 * o + 1] = im;
            kn[o] = cnt;
            reach_bad[o] = bad;
            if (want_exact) {
                const double hr_ = (double)er, hi_ = (double)ei;
                exact_hi[2 * o] = hr_;
                exact_hi[2 * o + 1] = hi_;
                exact_lo[2 * o] = (double)(er - hr_);
                exact_lo[2 * o + 1] = (double)(ei - hi_);
                const __float128 dr = (__float128)re - er, di = (__float128)im - ei;
                err[o] = (double)sqrtq(dr * dr + di * di);
                amag[o] = (double)a;
            }
        }
    }
    return (long)out0;
}
