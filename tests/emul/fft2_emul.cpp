// CPU emulation of the FFT v2 device code (comms-rs_b200/csrc/fft2_core.cuh): every pass is run for
// every thread of a frame in turn (a pass boundary = __syncthreads), with ping-pong shared-memory
// buffers, and the result is compared with an O(N^2) DFT in double.  Also reports the worst
// shared-memory bank-conflict degree per half-warp (8-byte words, 16 banks of 8 bytes).
// Build: g++ -O2 -std=c++17 -I/usr/local/cuda/include fft2_emul.cpp -o fft2_emul
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <vector>

#include "../../comms-rs_b200/csrc/fft2_core.cuh"

using namespace cb::fft2;

struct LogSm {
    float2 *base;
    std::vector<std::vector<int>> *log;  // [thread] -> sequence of padded indices
    int tid;
    float2 ld(int i) const { (*log)[tid].push_back(pad16(i)); return base[pad16(i)]; }
    void st(int i, float2 v) const { (*log)[tid].push_back(pad16(i)); base[pad16(i)] = v; }
};

static int worst_conflict(const std::vector<std::vector<int>> &log, int T)
{
    int worst = 1;
    if (log.empty() || log[0].empty()) return 0;
    const size_t nacc = log[0].size();
    for (size_t a = 0; a < nacc; ++a)
        for (int h0 = 0; h0 < T; h0 += 16) {
            std::map<int, std::vector<int>> banks;
            for (int t = h0; t < h0 + 16 && t < T; ++t) {
                const int w = log[t][a];
                auto &v = banks[w % 16];
                bool seen = false;
                for (int x : v) seen |= (x == w);
                if (!seen) v.push_back(w);
            }
            for (auto &kv : banks) worst = std::max(worst, (int)kv.second.size());
        }
    return worst;
}

template <int LOG2N, bool INV>
static void make_tw(std::vector<float2> &tw)
{
    using PL = Plan<LOG2N>;
    tw.assign(PL::TW_TOTAL > 0 ? PL::TW_TOTAL : 1, make_float2(0, 0));
    const long double sgn = INV ? 2.0L : -2.0L, pi = 3.14159265358979323846264338327950288L;
    for (int p = 1; p < PL::P16; ++p) {
        const int Ns = 1 << (4 * p);
        for (int s = 0; s < Ns; ++s) {
            const long double a = sgn * pi * s / (16.0L * Ns);
            tw[PL::tw_off(p) + s] = make_float2((float)cosl(a), (float)sinl(a));
        }
    }
    if (PL::REM) {
        const int n = PL::N >> PL::REM;
        for (int s = 0; s < n; ++s) {
            const long double a = sgn * pi * s / PL::N;
            tw[PL::tw_off(PL::P16) + s] = make_float2((float)cosl(a), (float)sinl(a));
        }
    }
}

template <int LOG2N, bool INV, int PASS>
static void emul_pass(const std::vector<float2> &x, std::vector<float2> &out, std::vector<float2> *buf,
                      const std::vector<float2> &tw, int &worst)
{
    using PL = Plan<LOG2N>;
    if constexpr (PASS < PL::PASSES) {
        std::vector<std::vector<int>> lin(PL::T), lout(PL::T);
        for (int j = 0; j < PL::T; ++j) {
            auto gld = [&](int i) { return x[i]; };
            auto gst = [&](int i, float2 v) { out[i] = v; };
            LogSm sin{buf[(PASS + 1) & 1].data(), &lin, j}, sout{buf[PASS & 1].data(), &lout, j};
            auto mid = [] {};
            run_pass<LOG2N, INV, PASS>(j, tw.data(), gld, gst, sin, sout, mid);
        }
        // loads and stores are logged separately (different buffers)
        worst = std::max(worst, worst_conflict(lin, PL::T));
        worst = std::max(worst, worst_conflict(lout, PL::T));
        emul_pass<LOG2N, INV, PASS + 1>(x, out, buf, tw, worst);
    }
}

template <int LOG2N, bool INV>
static int check()
{
    using PL = Plan<LOG2N>;
    const int N = PL::N;
    std::vector<float2> x(N), out(N), tw;
    srand(1234 + LOG2N);
    for (auto &v : x) v = make_float2(rand() / (float)RAND_MAX * 2 - 1, rand() / (float)RAND_MAX * 2 - 1);
    make_tw<LOG2N, INV>(tw);
    std::vector<float2> buf[2] = {std::vector<float2>(PL::PADN + 16), std::vector<float2>(PL::PADN + 16)};
    int worst = 0;
    emul_pass<LOG2N, INV, 0>(x, out, buf, tw, worst);
    // reference: direct DFT in double on a subset of bins (all bins for N <= 2048)
    const int step = N <= 2048 ? 1 : 7;
    double num = 0, den = 0;
    const double sgn = INV ? 1.0 : -1.0;
    for (int k = 0; k < N; k += step) {
        std::complex<double> acc = 0;
        for (int n = 0; n < N; ++n) {
            const double a = sgn * 2.0 * M_PI * (double)(((long long)k * n) % N) / N;
            acc += std::complex<double>(x[n].x, x[n].y) * std::complex<double>(cos(a), sin(a));
        }
        const std::complex<double> got(out[k].x, out[k].y);
        num += std::norm(got - acc);
        den += std::norm(acc);
    }
    const double rel = sqrt(num / den);
    printf("fft2 emul N=%5d inv=%d passes=%d rel_l2=%.3e worst_bank_conflict=%d %s\n", N, (int)INV, PL::PASSES, rel,
           worst, rel < 2e-6 ? "OK" : "FAIL");
    return rel < 2e-6 ? 0 : 1;
}

// ------------------------------------------------------------------ error ratios for tests/bounds.py
// Per frame: bin = max_k |got_k - X_k| / (u log2N S), S = sum |x_n|, and norm = ||got - X||_2 / (u log2N ||X||_2),
// u = 2^-24, X the transform in double.  Inputs: an impulse at every position (N <= 4096; digit / tile edges and
// pseudo-random positions above), tones on exact bins, and random frames, both directions.  The host arithmetic is
// the device's without FMA contraction (one more rounding per product): an upper estimate of its rounding error.
struct PlainSm {
    float2 *base;
    float2 ld(int i) const { return base[pad16(i)]; }
    void st(int i, float2 v) const { base[pad16(i)] = v; }
};

typedef std::complex<double> cd;

static void ref_fft(std::vector<cd> &a, bool inv)  // radix 2 in double, every twiddle from its exact angle
{
    const size_t n = a.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) std::swap(a[i], a[j]);
    }
    const long double pi = 3.14159265358979323846264338327950288L;
    for (size_t len = 2; len <= n; len <<= 1)
        for (size_t k = 0; k < len / 2; ++k) {
            const long double ang = (inv ? 2.0L : -2.0L) * pi * (long double)k / (long double)len;
            const cd w((double)cosl(ang), (double)sinl(ang));
            for (size_t i = 0; i < n; i += len) {
                const cd b = a[i + k + len / 2] * w;
                a[i + k + len / 2] = a[i + k] - b;
                a[i + k] += b;
            }
        }
}

struct Worst {
    double bin = 0, norm = 0;
};

static void ratios(const std::vector<float2> &x, const std::vector<float2> &got, bool inv, Worst &w)
{
    const int n = (int)x.size();
    int log2n = 0;
    while ((1 << log2n) < n) ++log2n;
    std::vector<cd> X(n);
    double S = 0;
    for (int i = 0; i < n; ++i) {
        X[i] = cd(x[i].x, x[i].y);
        S += std::abs(X[i]);
    }
    ref_fft(X, inv);
    const double u = std::ldexp(1.0, -24);
    double emax = 0, e2 = 0, x2 = 0;
    for (int k = 0; k < n; ++k) {
        const double e = std::abs(cd(got[k].x, got[k].y) - X[k]);
        emax = std::max(emax, e);
        e2 += e * e;
        x2 += std::norm(X[k]);
    }
    w.bin = std::max(w.bin, emax / (u * log2n * S));
    w.norm = std::max(w.norm, std::sqrt(e2 / x2) / (u * log2n));
}

template <int LOG2N, bool INV, int PASS>
static void plain_passes(const std::vector<float2> &x, std::vector<float2> &out, std::vector<float2> *buf,
                         const std::vector<float2> &tw)
{
    using PL = Plan<LOG2N>;
    if constexpr (PASS < PL::PASSES) {
        for (int j = 0; j < PL::T; ++j) {
            auto gld = [&](int i) { return x[i]; };
            auto gst = [&](int i, float2 v) { out[i] = v; };
            PlainSm sin{buf[(PASS + 1) & 1].data()}, sout{buf[PASS & 1].data()};
            auto mid = [] {};
            run_pass<LOG2N, INV, PASS>(j, tw.data(), gld, gst, sin, sout, mid);
        }
        plain_passes<LOG2N, INV, PASS + 1>(x, out, buf, tw);
    }
}

// 65536 = 256 x 256 as fft_rows_kernel.cu computes it: per column n2, two radix-16 passes (the second after
// twiddle16 by W_256^j); per row k1, twiddle16c by W_N^{k1 (lo + 16 m)}, radix 16, twiddle16 by W_256^hi, radix 16
template <bool INV>
static void rows65536(const std::vector<float2> &x, std::vector<float2> &out, const std::vector<float2> &twN)
{
    std::vector<float2> mid(65536), r(256);
    float2 v[16];
    for (int n2 = 0; n2 < 256; ++n2) {
        for (int j = 0; j < 16; ++j) {
            for (int m = 0; m < 16; ++m) v[m] = x[n2 + 256 * (j + 16 * m)];
            bfly16<INV>(v);
            for (int sl = 0; sl < 16; ++sl) r[16 * j + q16(sl)] = v[sl];
        }
        for (int j = 0; j < 16; ++j) {
            for (int m = 0; m < 16; ++m) v[m] = r[j + 16 * m];
            twiddle16(v, twN[256 * j]);
            bfly16<INV>(v);
            for (int sl = 0; sl < 16; ++sl) mid[256 * (j + 16 * q16(sl)) + n2] = v[sl];
        }
    }
    for (int k1 = 0; k1 < 256; ++k1) {
        for (int lo = 0; lo < 16; ++lo) {
            for (int m = 0; m < 16; ++m) v[m] = mid[256 * k1 + lo + 16 * m];
            twiddle16c(v, twN[k1 * lo], twN[16 * k1]);
            bfly16<INV>(v);
            for (int sl = 0; sl < 16; ++sl) r[16 * lo + q16(sl)] = v[sl];
        }
        for (int hi = 0; hi < 16; ++hi) {
            for (int m = 0; m < 16; ++m) v[m] = r[hi + 16 * m];
            twiddle16(v, twN[256 * hi]);
            bfly16<INV>(v);
            for (int sl = 0; sl < 16; ++sl) out[k1 + 256 * (hi + 16 * q16(sl))] = v[sl];
        }
    }
}

// frames of each kind for an N-point transform `run`
template <typename RUN>
static void sweep(int n, bool inv, RUN run, const char *what)
{
    Worst wi, wt, wr;
    std::vector<float2> x(n), out(n);
    std::vector<int> pos;
    if (n <= 4096) {
        for (int p = 0; p < n; ++p) pos.push_back(p);
    } else {
        for (int p : {0, 1, 15, 16, 17, 255, 256, 257, 4095, 4096, n / 2 - 1, n / 2, n - 16, n - 1}) pos.push_back(p);
        srand(77 + n);
        for (int i = 0; i < 48; ++i) pos.push_back(rand() % n);
    }
    for (int p : pos) {
        std::fill(x.begin(), x.end(), make_float2(0, 0));
        x[p] = make_float2(1, 0);
        run(x, out);
        ratios(x, out, inv, wi);
    }
    const long double pi = 3.14159265358979323846264338327950288L;
    for (int k0 : {1, 3, n / 4 + 1, n / 2 - 1, n - 5, (n * 5) / 7}) {
        for (int i = 0; i < n; ++i) {
            const long double a = 2.0L * pi * (long double)(((long long)k0 * i) % n) / n;
            x[i] = make_float2((float)cosl(a), (float)sinl(a));
        }
        run(x, out);
        ratios(x, out, inv, wt);
    }
    srand(1234 + n);
    for (int f = 0; f < 8; ++f) {
        for (auto &v : x) v = make_float2(rand() / (float)RAND_MAX * 2 - 1, rand() / (float)RAND_MAX * 2 - 1);
        run(x, out);
        ratios(x, out, inv, wr);
    }
    printf("fft2 ratio %s N=%d inv=%d impulse_bin=%.4f impulse_norm=%.4f tone_bin=%.4f tone_norm=%.4f random_bin=%.4f "
           "random_norm=%.4f\n",
           what, n, (int)inv, wi.bin, wi.norm, wt.bin, wt.norm, wr.bin, wr.norm);
}

template <int LOG2N, bool INV>
static void sweep_frames()
{
    using PL = Plan<LOG2N>;
    std::vector<float2> tw;
    make_tw<LOG2N, INV>(tw);
    std::vector<float2> buf[2] = {std::vector<float2>(PL::PADN + 16), std::vector<float2>(PL::PADN + 16)};
    sweep(PL::N, INV, [&](const std::vector<float2> &x, std::vector<float2> &out) { plain_passes<LOG2N, INV, 0>(x, out, buf, tw); },
          "frames");
}

template <bool INV>
static void sweep_rows65536()
{
    std::vector<float2> twN(65536);  // upload_twiddles (api.cu)
    const long double pi = 3.14159265358979323846264338327950288L;
    for (int k = 0; k < 65536; ++k) {
        const long double a = (INV ? 2.0L : -2.0L) * pi * k / 65536.0L;
        twN[k] = make_float2((float)cosl(a), (float)sinl(a));
    }
    sweep(65536, INV, [&](const std::vector<float2> &x, std::vector<float2> &out) { rows65536<INV>(x, out, twN); }, "rows");
}

// Chirp-z with M <= 16384 as bluestein_frames_kernel computes it (fft_kernels.cu): stage 0 loads x_i w_i (zero for
// i >= N) into the forward M-point passes and stores the product with B; stage 1 runs the inverse passes and stores
// (v w_k) 1/M for k < N.  The chirp w and B = the M-point transform of the wrapped conj chirp are built as
// bluestein_setup (api.cu) builds them: angles of i^2 mod 2N, B in double, both rounded to f32.  Ratios against the
// exact N-point transform: bin = max |err_k| / (u log2(M) S), norm = ||err|| / (u log2(M) ||X||).
template <int LOG2M>
static void sweep_chirpz(int n, bool inv)
{
    using PL = Plan<LOG2M>;
    const int M = PL::N;
    const long double pi = 3.14159265358979323846264338327950288L;
    std::vector<float2> w(n), bs(M), twf, twi;
    std::vector<cd> b(M, cd(0, 0));
    for (int i = 0; i < n; ++i) {
        const unsigned long long q = ((unsigned long long)i * i) % (2ull * n);
        const long double a = (inv ? 1.0L : -1.0L) * pi * (long double)q / (long double)n;
        w[i] = make_float2((float)cosl(a), (float)sinl(a));
        b[i] = cd((double)cosl(a), -(double)sinl(a));
        if (i) b[M - i] = b[i];
    }
    ref_fft(b, false);
    for (int i = 0; i < M; ++i) bs[i] = make_float2((float)b[i].real(), (float)b[i].imag());
    make_tw<LOG2M, false>(twf);
    make_tw<LOG2M, true>(twi);
    std::vector<float2> buf[2] = {std::vector<float2>(PL::PADN + 16), std::vector<float2>(PL::PADN + 16)};
    std::vector<float2> a(M), spec(M), c(M), out(n);
    std::vector<cd> tab(n);  // e^{-/+ 2 pi i s / N}
    for (int s = 0; s < n; ++s) {
        const long double ang = (inv ? 2.0L : -2.0L) * pi * (long double)s / (long double)n;
        tab[s] = cd((double)cosl(ang), (double)sinl(ang));
    }
    const float scale = 1.0f / (float)M;
    const double u = std::ldexp(1.0, -24);
    double wbin = 0, wnorm = 0;
    auto frame = [&](const std::vector<float2> &x) {
        for (int i = 0; i < M; ++i) a[i] = i < n ? cmul(x[i], w[i]) : make_float2(0, 0);
        plain_passes<LOG2M, false, 0>(a, spec, buf, twf);
        for (int i = 0; i < M; ++i) spec[i] = cmul(spec[i], bs[i]);
        plain_passes<LOG2M, true, 0>(spec, c, buf, twi);
        for (int k = 0; k < n; ++k) {
            const float2 r = cmul(c[k], w[k]);
            out[k] = make_float2(r.x * scale, r.y * scale);
        }
        double S = 0, e2 = 0, x2 = 0, emax = 0;
        std::vector<int> nz;
        for (int i = 0; i < n; ++i) {
            S += std::abs(cd(x[i].x, x[i].y));
            if (x[i].x != 0 || x[i].y != 0) nz.push_back(i);
        }
        for (int k = 0; k < n; ++k) {
            cd acc = 0;
            for (int i : nz) acc += cd(x[i].x, x[i].y) * tab[((long long)k * i) % n];
            const double e = std::abs(cd(out[k].x, out[k].y) - acc);
            emax = std::max(emax, e);
            e2 += e * e;
            x2 += std::norm(acc);
        }
        wbin = std::max(wbin, emax / (u * LOG2M * S));
        wnorm = std::max(wnorm, std::sqrt(e2 / x2) / (u * LOG2M));
    };
    std::vector<float2> x(n);
    std::vector<int> pos;
    if (n <= 1024) {
        for (int p = 0; p < n; ++p) pos.push_back(p);
    } else {
        for (int p : {0, 1, 2, n / 2, n - 2, n - 1}) pos.push_back(p);
        srand(99 + n);
        for (int i = 0; i < 26; ++i) pos.push_back(rand() % n);
    }
    for (int p : pos) {
        std::fill(x.begin(), x.end(), make_float2(0, 0));
        x[p] = make_float2(1, 0);
        frame(x);
    }
    for (int k0 : {1, n / 3 + 1, n - 2}) {
        for (int i = 0; i < n; ++i) {
            const long double ang = 2.0L * pi * (long double)(((long long)k0 * i) % n) / n;
            x[i] = make_float2((float)cosl(ang), (float)sinl(ang));
        }
        frame(x);
    }
    srand(4321 + n);
    for (int f = 0; f < 3; ++f) {
        for (auto &v : x) v = make_float2(rand() / (float)RAND_MAX * 2 - 1, rand() / (float)RAND_MAX * 2 - 1);
        frame(x);
    }
    printf("chirpz ratio N=%d M=%d inv=%d bin=%.4f norm=%.4f\n", n, M, (int)inv, wbin, wnorm);
}

template <int LOG2N>
static void sweep_both()
{
    sweep_frames<LOG2N, false>();
    sweep_frames<LOG2N, true>();
}

int main()
{
    sweep_both<4>();
    sweep_both<5>();
    sweep_both<6>();
    sweep_both<7>();
    sweep_both<8>();
    sweep_both<9>();
    sweep_both<10>();
    sweep_both<11>();
    sweep_both<12>();
    sweep_both<13>();
    sweep_both<14>();
    sweep_rows65536<false>();
    sweep_rows65536<true>();
    for (int inv = 0; inv < 2; ++inv) {  // every fused chirp-z size class up to M = 16384
        sweep_chirpz<9>(129, inv);
        sweep_chirpz<11>(1000, inv);
        sweep_chirpz<13>(4095, inv);
        sweep_chirpz<14>(4097, inv);
        sweep_chirpz<14>(8191, inv);
    }
    int bad = 0;
    bad += check<4, false>();
    bad += check<5, false>();
    bad += check<6, true>();
    bad += check<7, false>();
    bad += check<8, false>();
    bad += check<8, true>();
    bad += check<9, false>();
    bad += check<10, false>();
    bad += check<10, true>();
    bad += check<11, false>();
    bad += check<12, false>();
    bad += check<12, true>();
    bad += check<13, false>();
    bad += check<14, true>();  // the largest one-CTA size (4 passes: 16 16 16 4)
    return bad;
}
