// Complex<f64> FFT (cb_fft_f64): the arithmetic every f64 transform path shares, as host/device code, and the host
// tables.  The kernels (fft_f64_kernels.cu) and the CPU emulation (tests/emul/fft_f64_emul.cpp) both run these
// functions, so a butterfly, a twiddle product or a chirp product rounds identically on the device and in the
// emulation.  On the device every operation is an explicit __dadd_rn / __dmul_rn / __fma_rn; on the host it is a
// separately rounded + / * or std::fma, and the emulation is compiled with -ffp-contract=off so that nothing fuses.
//
// The tables are computed once on the host in long double (64-bit mantissa) and each value is rounded to double once:
// twiddles e^{-/+2 pi i m / n} with the angle reduced to [-pi/4, pi/4] in integers (so quarter turns are exact), the
// chirp e^{-/+ i pi q / N} with q = i^2 mod 2N formed in integers, and the chirp spectrum by a long-double FFT.
#pragma once
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

#ifdef __CUDACC__
#define F64_HD __host__ __device__ __forceinline__
#else
#define F64_HD inline
#endif

namespace cb {
namespace f64fft {

struct alignas(16) z64 {
    double re, im;
};

F64_HD double dadd(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
F64_HD double dsub(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
F64_HD double dmul(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
F64_HD double dfma(double a, double b, double c)
{
#ifdef __CUDA_ARCH__
    return __fma_rn(a, b, c);
#else
    return std::fma(a, b, c);
#endif
}

F64_HD z64 cadd(z64 a, z64 b) { return {dadd(a.re, b.re), dadd(a.im, b.im)}; }
F64_HD z64 csub(z64 a, z64 b) { return {dsub(a.re, b.re), dsub(a.im, b.im)}; }
// a * w: re = fma(a.re, w.re, -(a.im w.im)), im = fma(a.re, w.im, a.im w.re) -- one product rounded, one fused
F64_HD z64 cmul(z64 a, z64 w)
{
    const double t = dmul(a.im, w.im), s = dmul(a.im, w.re);
    return {dfma(a.re, w.re, -t), dfma(a.re, w.im, s)};
}
// a * (-/+ i): exact
template <bool INV>
F64_HD z64 cmul_i(z64 a)
{
    return INV ? z64{-a.im, a.re} : z64{a.im, -a.re};
}

// sqrt(1/2) rounded to double
constexpr double SQRT1_2 = 0.70710678118654752440;

// a * e^{-/+ i pi/4} = c ((a.re + a.im) + i (a.im - a.re)) forward, c ((a.re - a.im) + i (a.im + a.re)) inverse
template <bool INV>
F64_HD z64 cmul_w8(z64 a)
{
    const double s = INV ? dsub(a.re, a.im) : dadd(a.re, a.im);
    const double d = INV ? dadd(a.im, a.re) : dsub(a.im, a.re);
    return {dmul(s, SQRT1_2), dmul(d, SQRT1_2)};
}
// a * e^{-/+ 3 i pi/4} = c ((a.im - a.re) - i (a.re + a.im)) forward, c (-(a.re + a.im) + i (a.re - a.im)) inverse
template <bool INV>
F64_HD z64 cmul_w83(z64 a)
{
    const double s = dadd(a.re, a.im), d = INV ? dsub(a.re, a.im) : dsub(a.im, a.re);
    return INV ? z64{-dmul(s, SQRT1_2), dmul(d, SQRT1_2)} : z64{dmul(d, SQRT1_2), -dmul(s, SQRT1_2)};
}

// In-place DFT of R = 2, 4 or 8 points in natural order, e^{-/+ 2 pi i jk / R}: radix-2 decimation in frequency.
// Only additions, exact multiplications by -/+ i and, for R = 8, the two e^{-/+ i pi/4} products above round.
template <int R, bool INV>
F64_HD void dft(z64 *v)
{
    if (R == 2) {
        const z64 a = v[0], b = v[1];
        v[0] = cadd(a, b);
        v[1] = csub(a, b);
    } else if (R == 4) {
        const z64 b0 = cadd(v[0], v[2]), b2 = csub(v[0], v[2]);
        const z64 b1 = cadd(v[1], v[3]), b3 = cmul_i<INV>(csub(v[1], v[3]));
        v[0] = cadd(b0, b1);
        v[2] = csub(b0, b1);
        v[1] = cadd(b2, b3);
        v[3] = csub(b2, b3);
    } else {
        z64 u[4], w[4];
        u[0] = cadd(v[0], v[4]);
        w[0] = csub(v[0], v[4]);
        u[1] = cadd(v[1], v[5]);
        w[1] = cmul_w8<INV>(csub(v[1], v[5]));
        u[2] = cadd(v[2], v[6]);
        w[2] = cmul_i<INV>(csub(v[2], v[6]));
        u[3] = cadd(v[3], v[7]);
        w[3] = cmul_w83<INV>(csub(v[3], v[7]));
        dft<4, INV>(u);
        dft<4, INV>(w);
        for (int m = 0; m < 4; ++m) {
            v[2 * m] = u[m];
            v[2 * m + 1] = w[m];
        }
    }
}

// One Stockham butterfly of a radix-R pass at stride p (p = 1, R, R^2, ... in points of the n-point sub-transform):
// butterfly i (0 <= i < n / R) reads v[j] = x[i + j n / R], multiplies v[j] (j >= 1) by tw[j k m] with k = i mod p and
// m = tw_step * n / (p R) (tw is a table of e^{-/+ 2 pi i e / NT}, NT = tw_step * n), takes the R-point DFT and writes
// v[j] to y[(i - k) R + k + j p].  k = 0 multiplies by nothing (the twiddles are exactly 1).
template <int R, bool INV>
F64_HD void stockham_bfly(z64 *v, const z64 *tw, unsigned k, unsigned m)
{
    if (k)
        for (int j = 1; j < R; ++j) v[j] = cmul(v[j], tw[(size_t)j * k * m]);
    dft<R, INV>(v);
}

// One term of a direct sum X[k] += x[n] tw[kn mod N]: two FMA chains, real and imaginary part.
F64_HD z64 direct_term(z64 acc, z64 x, z64 w)
{
    acc.re = dfma(x.re, w.re, acc.re);
    acc.re = dfma(-x.im, w.im, acc.re);
    acc.im = dfma(x.re, w.im, acc.im);
    acc.im = dfma(x.im, w.re, acc.im);
    return acc;
}

// ------------------------------------------------------------------------------------------------- host tables
// e^{sgn 2 pi i a / b}, 0 <= a < b, correctly reduced: the nearest quarter turn q and the residue r = 4a - q b are
// integers, the residual angle pi r / (2 b) is in [-pi/4, pi/4], and the quarter turn is applied exactly.
inline z64 unit_ld(uint64_t a, uint64_t b, int sgn)
{
    const long double PI_L = 3.14159265358979323846264338327950288L;
    const uint64_t q = (4 * a + b / 2) / b;
    const long long r = (long long)(4 * a) - (long long)(q * b);
    const long double t = PI_L * (long double)r / (2.0L * (long double)b);
    long double c = r ? cosl(t) : 1.0L, s = r ? sinl(t) : 0.0L;
    for (uint64_t j = 0; j < (q & 3); ++j) {
        const long double c2 = -s;
        s = c;
        c = c2;
    }
    return {(double)c, sgn < 0 ? -(double)s : (double)s};
}

// tw[e] = e^{-/+ 2 pi i e / n}, e < n ("+" when inverse)
inline std::vector<z64> twiddle_table(size_t n, int inverse)
{
    std::vector<z64> t(n);
    for (size_t e = 0; e < n; ++e) t[e] = unit_ld(e, n, inverse ? 1 : -1);
    return t;
}

// Chirp-z tables for N points padded to M (a power of two >= 2N - 1):
//   chirp[i] = e^{-/+ i pi q / N}, q = i^2 mod 2N  (i < N)
//   bspec[j] = (1/M) sum_i b[i] e^{-2 pi i j i / M}, b[i] = conj(chirp[|i|]) at i and M - i (|i| < N), else 0,
// the spectrum by a radix-2 FFT in long double over long-double twiddles, rounded to double once (the 1/M of the
// inverse transform is folded in, exactly: M is a power of two).
inline void chirp_tables(size_t N, size_t M, int inverse, std::vector<z64> &chirp, std::vector<z64> &bspec)
{
    const long double PI_L = 3.14159265358979323846264338327950288L;
    chirp.resize(N);
    std::vector<long double> br(M, 0.0L), bi(M, 0.0L);
    for (size_t i = 0; i < N; ++i) {
        const unsigned long long q = ((unsigned long long)i * i) % (2ull * N);
        // q / N = 2 q / 2N: the same reduced angle as a twiddle of 2N points
        chirp[i] = unit_ld(q, 2 * N, inverse ? 1 : -1);
        const long double a = (inverse ? 1.0L : -1.0L) * PI_L * (long double)q / (long double)N;
        br[i] = cosl(a);
        bi[i] = -sinl(a);
        if (i) {
            br[M - i] = br[i];
            bi[M - i] = bi[i];
        }
    }
    // forward radix-2 FFT in long double, twiddles e^{-2 pi i e / M} from one table
    std::vector<long double> wr(M / 2), wi(M / 2);
    for (size_t e = 0; e < M / 2; ++e) {
        const long double a = -2.0L * PI_L * (long double)e / (long double)M;
        wr[e] = cosl(a);
        wi[e] = sinl(a);
    }
    for (size_t i = 1, j = 0; i < M; ++i) {
        size_t bit = M >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) {
            std::swap(br[i], br[j]);
            std::swap(bi[i], bi[j]);
        }
    }
    for (size_t len = 2; len <= M; len <<= 1) {
        const size_t half = len >> 1, step = M / len;
        for (size_t i = 0; i < M; i += len)
            for (size_t k = 0; k < half; ++k) {
                const long double c = wr[k * step], s = wi[k * step];
                const long double xr = br[i + k + half] * c - bi[i + k + half] * s;
                const long double xi = br[i + k + half] * s + bi[i + k + half] * c;
                br[i + k + half] = br[i + k] - xr;
                bi[i + k + half] = bi[i + k] - xi;
                br[i + k] += xr;
                bi[i + k] += xi;
            }
    }
    bspec.resize(M);
    for (size_t j = 0; j < M; ++j) bspec[j] = {(double)(br[j] / (long double)M), (double)(bi[j] / (long double)M)};
}

// ------------------------------------------------------------------------------------------------- plan shape
// Powers of two from 8 to FRAME_MAX points: one frame kernel launch.  Larger powers of two up to 2^20: two steps of
// N1 x N2 = N points (N1 = 2^floor(L/2) <= N2 = 2^ceil(L/2) <= 1024).  Other lengths up to DIRECT_MAX, and 1, 2, 4:
// direct sums.  Anything else up to 2^19: chirp-z over M = the least power of two >= max(8, 2N - 1).
constexpr unsigned FRAME_MAX_LOG2 = 12;
constexpr size_t DIRECT_MAX = 128;
constexpr unsigned CTA_POINTS = 2048;  // points per CTA of the frame / column kernel when a sub-transform is smaller

// columns per CTA: sub-transforms of n points, with the CTA's strided side contiguous over the columns (col_major)
inline unsigned cols_per_cta(unsigned log2n, bool col_major)
{
    const unsigned n = 1u << log2n, b = n >= CTA_POINTS ? 1u : CTA_POINTS / n;
    return col_major && b < 4 ? 4u : b;
}

}  // namespace f64fft
}  // namespace cb
