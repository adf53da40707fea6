// CPU emulation of the Complex<f64> FFT (include/comms_b200.h, cb_fft_f64): every path of the plan, butterfly by
// butterfly, through the same host/device functions the kernels run (comms-rs_b200/csrc/fft64_core.cuh) and the same
// host tables.  Built as a shared library (g++ -O2 -std=c++17 -ffp-contract=off -fopenmp -shared -fPIC) and called
// through ctypes by tests/test_fft_f64_cpu.py and tests/test_gpu_fft_f64.py.
//
// `mutation` != 0 reproduces one defect the tests must reject (see the enum).
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

#include "../../comms-rs_b200/csrc/fft64_core.cuh"

using namespace cb::f64fft;

namespace {

enum Mutation {
    NONE = 0,
    TW_F32 = 1,         // one twiddle (j = 1, k = 1) of the second Stockham pass carried at f32 precision
    BIN_ULP = 2,        // the largest bin of every frame off by 2^16 ulp
    CHIRP_ANGLE = 3,    // the chirp angle formed as pi i^2 / N in double, without the integer reduction
    CHIRP_SPEC_F64 = 4, // the chirp spectrum from a radix-2 FFT in double instead of long double
    NAN_LEAK = 5,       // a non-finite chirp-z frame leaks a NaN into the next frame of its group
    INV_FWD_TW = 6,     // the inverse plan multiplies by forward twiddles in its last pass
};

// one butterfly, with the twiddles a mutation may alter
template <int R, bool INV>
void bfly(z64 *v, const z64 *tw, unsigned k, unsigned m, int mutation, unsigned pass, bool last)
{
    if (!((mutation == TW_F32 && pass == 1 && k == 1) || (mutation == INV_FWD_TW && INV && last))) {
        stockham_bfly<R, INV>(v, tw, k, m);
        return;
    }
    if (k)
        for (int j = 1; j < R; ++j) {
            z64 w = tw[(size_t)j * k * m];
            if (mutation == TW_F32 && j == 1) w = {(double)(float)w.re, (double)(float)w.im};
            if (mutation == INV_FWD_TW) w.im = -w.im;
            v[j] = cmul(v[j], w);
        }
    dft<R, INV>(v);
}

template <int R, bool INV>
void pass(const z64 *x, z64 *y, unsigned n, unsigned p, const z64 *tw, unsigned tw_step, int mutation, unsigned ps,
          bool last)
{
    const unsigned nb = n / R, m = tw_step * (n / (p * R));
    for (unsigned i = 0; i < nb; ++i) {
        const unsigned k = i & (p - 1);
        z64 v[R];
        for (int j = 0; j < R; ++j) v[j] = x[i + j * nb];
        bfly<R, INV>(v, tw, k, m, mutation, ps, last);
        for (int j = 0; j < R; ++j) y[(i - k) * R + k + j * p] = v[j];
    }
}

// the frame kernel's passes over one contiguous column of 2^L points (L >= 3), in place
template <bool INV>
void sub_fft(z64 *x, unsigned L, const z64 *tw, unsigned tw_step, int mutation)
{
    const unsigned n = 1u << L, n8 = L / 3, rem = L % 3, np = n8 + (rem ? 1 : 0);
    std::vector<z64> buf(n);
    z64 *a = x, *b = buf.data();
    unsigned p = 1, ps = 0;
    for (; ps < n8; ++ps, p *= 8) {
        pass<8, INV>(a, b, n, p, tw, tw_step, mutation, ps, ps + 1 == np);
        std::swap(a, b);
    }
    if (rem == 2) pass<4, INV>(a, b, n, p, tw, tw_step, mutation, ps, true), std::swap(a, b);
    if (rem == 1) pass<2, INV>(a, b, n, p, tw, tw_step, mutation, ps, true), std::swap(a, b);
    if (a != x)
        for (unsigned e = 0; e < n; ++e) x[e] = a[e];
}

// one frame of 2^L points: the frame kernel, or the two steps with the inter-step twiddle tw[k1 n2]
template <bool INV>
void pow2_frame(const z64 *x, z64 *y, unsigned L, const z64 *tw, int mutation)
{
    const size_t N = (size_t)1 << L;
    if (L <= FRAME_MAX_LOG2) {
        for (size_t e = 0; e < N; ++e) y[e] = x[e];
        sub_fft<INV>(y, L, tw, 1, mutation);
        return;
    }
    const unsigned L1 = L / 2, L2 = L - L1;
    const size_t N1 = (size_t)1 << L1, N2 = (size_t)1 << L2;
    std::vector<z64> mid(N), col(N1 > N2 ? N1 : N2);
    for (size_t n2 = 0; n2 < N2; ++n2) {
        for (size_t n1 = 0; n1 < N1; ++n1) col[n1] = x[n1 * N2 + n2];
        sub_fft<INV>(col.data(), L1, tw, (unsigned)N2, mutation);
        for (size_t k1 = 0; k1 < N1; ++k1) {
            const size_t t = k1 * n2;
            mid[n2 * N1 + k1] = t ? cmul(col[k1], tw[t]) : col[k1];
        }
    }
    for (size_t k1 = 0; k1 < N1; ++k1) {
        for (size_t n2 = 0; n2 < N2; ++n2) col[n2] = mid[n2 * N1 + k1];
        sub_fft<INV>(col.data(), L2, tw, (unsigned)N1, mutation);
        for (size_t k2 = 0; k2 < N2; ++k2) y[k1 + N1 * k2] = col[k2];
    }
}

void pow2_any(const z64 *x, z64 *y, unsigned L, const z64 *tw, int inverse, int mutation)
{
    if (inverse) pow2_frame<true>(x, y, L, tw, mutation);
    else pow2_frame<false>(x, y, L, tw, mutation);
}

// the f64 radix-2 host FFT an earlier chirp-z spectrum used (CHIRP_SPEC_F64)
void host_fft_double(std::vector<double> &re, std::vector<double> &im)
{
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) {
            std::swap(re[i], re[j]);
            std::swap(im[i], im[j]);
        }
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        const size_t half = len >> 1;
        for (size_t k = 0; k < half; ++k) {
            const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)k / (long double)len;
            const double wr = (double)cosl(a), wi = (double)sinl(a);
            for (size_t i = 0; i < n; i += len) {
                const double xr = re[i + k + half] * wr - im[i + k + half] * wi;
                const double xi = re[i + k + half] * wi + im[i + k + half] * wr;
                re[i + k + half] = re[i + k] - xr;
                im[i + k + half] = im[i + k] - xi;
                re[i + k] += xr;
                im[i + k] += xi;
            }
        }
    }
}

}  // namespace

// y = the plan's output for `frames` contiguous frames of n points (2 n frames doubles each way).  Returns the path:
// 0 direct, 1 frame kernel, 2 two-step, 3 chirp-z; -1 for an unsupported size.
extern "C" int fft64_emul(const double *xin, size_t n, size_t frames, int inverse, int mutation, double *yout)
{
    const z64 *x = reinterpret_cast<const z64 *>(xin);
    z64 *y = reinterpret_cast<z64 *>(yout);
    const bool pow2 = (n & (n - 1)) == 0;
    if (n == 0 || n > ((size_t)1 << (pow2 ? 20 : 19))) return -1;
    unsigned L = 0;
    while (((size_t)1 << L) < n) ++L;
    int path;
    if (pow2 && L >= 3) {
        path = L <= FRAME_MAX_LOG2 ? 1 : 2;
        const std::vector<z64> tw = twiddle_table(n, inverse);
#pragma omp parallel for schedule(dynamic)
        for (long long f = 0; f < (long long)frames; ++f) pow2_any(x + f * n, y + f * n, L, tw.data(), inverse, mutation);
    } else if (pow2 || n <= DIRECT_MAX) {
        path = 0;
        const std::vector<z64> tw = twiddle_table(n, inverse);
#pragma omp parallel for schedule(static)
        for (long long f = 0; f < (long long)frames; ++f)
            for (size_t k = 0; k < n; ++k) {
                z64 acc{0.0, 0.0};
                size_t e = 0;
                for (size_t t = 0; t < n; ++t) {
                    acc = direct_term(acc, x[f * n + t], tw[e]);
                    e += k;
                    if (e >= n) e -= n;
                }
                y[f * n + k] = acc;
            }
    } else {
        path = 3;
        size_t M = 8;
        while (M < 2 * n - 1) M <<= 1;
        unsigned LM = 0;
        while (((size_t)1 << LM) < M) ++LM;
        std::vector<z64> chirp, bspec;
        chirp_tables(n, M, inverse, chirp, bspec);
        if (mutation == CHIRP_ANGLE)
            for (size_t i = 0; i < n; ++i) {
                const double a = 3.141592653589793 * ((double)i * (double)i) / (double)n;
                chirp[i] = {std::cos(a), inverse ? std::sin(a) : -std::sin(a)};
            }
        if (mutation == CHIRP_SPEC_F64) {
            std::vector<double> br(M, 0.0), bi(M, 0.0);
            for (size_t i = 0; i < n; ++i) {
                br[i] = chirp[i].re;
                bi[i] = -chirp[i].im;
                if (i) {
                    br[M - i] = br[i];
                    bi[M - i] = bi[i];
                }
            }
            host_fft_double(br, bi);
            for (size_t j = 0; j < M; ++j) bspec[j] = {br[j] / (double)M, bi[j] / (double)M};
        }
        const std::vector<z64> twf = twiddle_table(M, 0), twi = twiddle_table(M, 1);
#pragma omp parallel for schedule(dynamic)
        for (long long f = 0; f < (long long)frames; ++f) {
            std::vector<z64> a(M), b(M);
            for (size_t t = 0; t < M; ++t) a[t] = t < n ? cmul(x[f * n + t], chirp[t]) : z64{0.0, 0.0};
            pow2_any(a.data(), b.data(), LM, twf.data(), 0, mutation == TW_F32 || mutation == INV_FWD_TW ? 0 : mutation);
            for (size_t j = 0; j < M; ++j) b[j] = cmul(b[j], bspec[j]);
            pow2_any(b.data(), a.data(), LM, twi.data(), 1, mutation == TW_F32 || mutation == INV_FWD_TW ? 0 : mutation);
            for (size_t k = 0; k < n; ++k) y[f * n + k] = cmul(a[k], chirp[k]);
        }
        if (mutation == NAN_LEAK)
            for (size_t f = 0; f + 1 < frames; ++f) {
                bool bad = false;
                for (size_t k = 0; k < n; ++k) bad |= !std::isfinite(y[f * n + k].re) || !std::isfinite(y[f * n + k].im);
                if (bad) y[(f + 1) * n].re = NAN;
            }
    }
    if (mutation == BIN_ULP)
        for (size_t f = 0; f < frames; ++f) {
            size_t best = 0;
            for (size_t k = 1; k < n; ++k)
                if (std::hypot(y[f * n + k].re, y[f * n + k].im) > std::hypot(y[f * n + best].re, y[f * n + best].im)) best = k;
            double &v = y[f * n + best].re;
            if (std::isfinite(v) && v != 0.0) v += std::ldexp(1.0, std::ilogb(v) - 52 + 16);
        }
    return path;
}
