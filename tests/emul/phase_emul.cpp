// CPU emulation of the device's f64 operation sequence in the NCO scan (nco_kernel.cu) and the two f64 estimators
// (estimator_kernels.cu), against references in __float128 / long double.  Built with g++ -O2 -ffp-contract=off; every
// fused multiply-add of the device is an explicit std::fma here, every other operation rounds on its own, and the
// thread, warp, CTA and chunk orders are those of the kernels at their real launch shapes.  The device's f64 sincos
// (2 ulp) is not emulated: the NCO ratios are of the phase before sincos, the estimator ratios of the complex sum.
//
//   phase_emul nco <old|fixed> <case> A B      worst ratio of |phase_k - phi_k| over u64 (A (|phase0| + 2 pi (1 +
//                                              chunks_k)) + B S_k), S_k = sum_{i<=k} |perr_i|, over every causal output
//   phase_emul freq <case> C                   |S_dev - S| / (C u64 D_F sum |x_{i+1}| |x_i|)
//   phase_emul timing <N> <D> <n> <case> C     |S_dev - S| / (C u64 (ntaps4 + D_T) sum |dout_i| A_i)
//
// "old" is the prefix order the NCO used before: exclusive prefixes formed as incl - v (tile scan) and incl - mine
// (in-tile scan).  One huge or non-finite perr_j then reaches the outputs before j.  "fixed" shifts the inclusive scans
// up one lane instead.  Each run prints one JSON line.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <quadmath.h>
#include <string>
#include <vector>

typedef __float128 f128;
static const double U64 = 0x1p-53;
static const double TWO_PI = 6.283185307179586476925;

static uint64_t rng_state = 0x9E3779B97F4A7C15ull;
static uint64_t next_u64()
{
    uint64_t z = (rng_state += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
static double uni() { return (double)(next_u64() >> 11) * 0x1p-53; }  // [0, 1)

// ------------------------------------------------------------------------------------------------------------- NCO
static const int NT = 256, PER = 8, TILE = NT * PER;

static double reduce_2pi(double hi, double lo)
{
    const double inv2pi = 0.15915494309189534561;
    const double C1 = 0x1.921fb40000000p+2, C2 = 0x1.4442d00000000p-22, C3 = 0x1.8469880000000p-46,
                 C4 = 0x1.8cc51701b839ap-70;
    const double q = std::nearbyint(hi * inv2pi);
    double r = std::fma(-q, C1, hi);
    r = std::fma(-q, C2, r);
    r = std::fma(-q, C3, r);
    r = std::fma(-q, C4, r);
    return r + lo;
}

// inclusive Hillis-Steele scan of 32 lanes (shfl_up by 1, 2, 4, 8, 16)
static void warp_scan(double *v)
{
    for (int o = 1; o < 32; o <<= 1) {
        double t[32];
        for (int l = 0; l < 32; ++l) t[l] = l >= o ? v[l - o] : 0.0;
        for (int l = o; l < 32; ++l) v[l] += t[l];
    }
}

static std::vector<double> nco_emul(const std::vector<double> &perr, double ph0, double dphase, bool old, double *phase_out)
{
    const size_t n = perr.size(), ntiles = (n + TILE - 1) / TILE;
    std::vector<double> tile(ntiles), ph(n);
    // nco_tile_sum_kernel: thread-sequential, xor butterfly, then warps 0..7 in order
    for (size_t b = 0; b < ntiles; ++b) {
        double ws[NT / 32];
        for (int w = 0; w < NT / 32; ++w) {
            double s[32];
            for (int l = 0; l < 32; ++l) {
                const size_t base = b * TILE + (size_t)(w * 32 + l) * PER;
                s[l] = 0.0;
                for (int i = 0; i < PER; ++i)
                    if (base + i < n) s[l] += perr[base + i];
            }
            for (int o = 16; o > 0; o >>= 1) {
                double t[32];
                for (int l = 0; l < 32; ++l) t[l] = s[l] + s[l ^ o];
                memcpy(s, t, sizeof s);
            }
            ws[w] = s[0];
        }
        double t = 0.0;
        for (int w = 0; w < NT / 32; ++w) t += ws[w];
        tile[b] = t;
    }
    // nco_scan_tiles_kernel: chunks of 1024 tile sums, carry reduced mod 2 pi
    double carry = 0.0;
    for (size_t c = 0; c < ntiles; c += 1024) {
        double v[1024], incl[1024], ws[32];
        for (int i = 0; i < 1024; ++i) v[i] = incl[i] = c + i < ntiles ? tile[c + i] : 0.0;
        for (int w = 0; w < 32; ++w) warp_scan(incl + 32 * w);
        for (int w = 0; w < 32; ++w) ws[w] = incl[32 * w + 31];
        warp_scan(ws);
        for (int i = 0; i < 1024; ++i) {
            const double before = (i >> 5) ? ws[(i >> 5) - 1] : 0.0;
            const double excl = old ? incl[i] - v[i] : ((i & 31) ? incl[i - 1] : 0.0);
            if (c + i < ntiles) tile[c + i] = reduce_2pi(carry + before + excl, 0.0);
        }
        carry = reduce_2pi(carry + ws[30] + incl[1023], 0.0);
    }
    // nco_apply_kernel
    for (size_t b = 0; b < ntiles; ++b) {
        double v[NT][PER], incl[NT], mine[NT], ws[NT / 32];
        for (int t = 0; t < NT; ++t) {
            const size_t base = b * TILE + (size_t)t * PER;
            for (int i = 0; i < PER; ++i) v[t][i] = base + i < n ? perr[base + i] : 0.0;
            for (int i = 1; i < PER; ++i) v[t][i] += v[t][i - 1];
            incl[t] = mine[t] = v[t][PER - 1];
        }
        for (int w = 0; w < NT / 32; ++w) warp_scan(incl + 32 * w);
        for (int w = 0; w < NT / 32; ++w) ws[w] = incl[32 * w + 31];
        for (int t = 0; t < NT; ++t) {
            const double excl = old ? incl[t] - mine[t] : ((t & 31) ? incl[t - 1] : 0.0);
            double off = tile[b] + excl;
            for (int w = 0; w < (t >> 5); ++w) off += ws[w];
            const size_t base = b * TILE + (size_t)t * PER;
            for (int i = 0; i < PER; ++i) {
                const size_t k = base + i;
                if (k >= n) break;
                const double kd = (double)(k + 1);
                const double hi = kd * dphase, lo = std::fma(kd, dphase, -hi);
                ph[k] = ph0 + reduce_2pi(hi, lo) + (off + v[t][i]);
                if (k == n - 1) {
                    double r = reduce_2pi(ph[k], 0.0);
                    if (r < 0.0) r += TWO_PI;
                    *phase_out = r;
                }
            }
        }
    }
    return ph;
}

static f128 wrap_q(f128 x)
{
    const f128 tp = (f128)6.283185307179586 + (f128)2.4492935982947064e-16 + (f128)-5.989539619436679e-33;  // 2 pi, 159 bits
    x -= tp * nearbyintq(x / tp);
    return x;
}

static int run_nco(const char *order, const std::string &cs, double A, double B)
{
    const bool old = !strcmp(order, "old");
    size_t n = 5000;
    double ph0 = 0.5, dphase = 0.37;
    size_t j = (size_t)-1;  // a non-finite perr
    std::vector<double> perr;
    if (cs == "phase0") {  // the |phase_0| term: ph0 + reduce + (off + v) rounds twice at |phase_0|
        ph0 = 1e6 + 0.3;
        n = 100000;
        perr.resize(n);
        for (auto &p : perr) p = std::ldexp(std::floor((uni() * 2 - 1) * 0x1p30), -40);
    } else if (cs == "random" || cs == "random3") {  // dyadic perr, |perr| < 2^-10, three scan chunks
        n = cs == "random" ? 100000 : 3 * (size_t)(1 << 21) + 7;
        dphase = TWO_PI - 0x1p-20;
        perr.resize(n);
        for (auto &p : perr) p = std::ldexp(std::floor((uni() * 2 - 1) * 0x1p30), -40);
    } else if (cs == "chain") {  // every addition of the thread-local scans rounds up by about u64
        ph0 = 0.0;
        dphase = 0.0;
        n = 4096;
        perr.resize(n);
        for (size_t k = 0; k < n; ++k) perr[k] = k % PER == 0 ? 1.0 : 0x1p-53 * (1 + 0x1p-20);
    } else if (cs == "huge" || cs == "nan") {  // one 1e6 or NaN in the middle of a thread, warp and tile
        n = 3 * TILE + 11;
        perr.resize(n);
        for (auto &p : perr) p = std::ldexp(std::floor((uni() * 2 - 1) * 0x1p30), -40);
        j = TILE + 1000 + 3;
        perr[j] = cs == "huge" ? 1e6 : NAN;
        if (cs == "huge") j = (size_t)-1;
    } else {
        fprintf(stderr, "unknown nco case %s\n", cs.c_str());
        return 2;
    }
    double pout = 0.0;
    const std::vector<double> ph = nco_emul(perr, ph0, dphase, old, &pout);
    f128 pre = 0;
    double S = 0.0, worst = 0.0;
    size_t wk = 0, nbad = 0, notnan = 0;
    for (size_t k = 0; k < n; ++k) {
        if (j != (size_t)-1 && k >= j) {
            notnan += !std::isnan(ph[k]);
            continue;
        }
        pre += (f128)perr[k];
        S += std::fabs(perr[k]);
        const f128 phi = (f128)ph0 + (f128)(double)(k + 1) * (f128)dphase + pre;
        const double err = std::isfinite(ph[k]) ? std::fabs((double)wrap_q((f128)ph[k] - phi)) : INFINITY;
        const double bound = U64 * (A * (std::fabs(ph0) + TWO_PI * (1 + (double)(k / (1024 * TILE)))) + B * S);
        const double r = err / bound;
        if (!(r <= 1.0)) ++nbad;
        if (!(r <= worst)) worst = r, wk = k;
    }
    if (j != (size_t)-1) notnan += !std::isnan(pout);
    printf("{\"kernel\": \"nco\", \"order\": \"%s\", \"case\": \"%s\", \"n\": %zu, \"worst\": %.6g, \"k\": %zu, "
           "\"outside\": %zu, \"not_nan_after\": %zu}\n",
           order, cs.c_str(), n, std::isfinite(worst) ? worst : 1e300, wk, nbad, notnan);
    return 0;
}

// -------------------------------------------------------------------------------------------------- estimators
struct c2 {
    double x, y;
};
static const unsigned MAXP = 148 * 8;

// block_sum: shfl_down tree over each warp, then thread 0 adds warps 1..7 in order
static c2 block_sum(std::vector<c2> v)
{
    for (int w = 0; w < NT / 32; ++w)
        for (int o = 16; o > 0; o >>= 1)
            for (int l = 0; l + o < 32; ++l) {  // lanes l < 32 - o read lane l + o's value before it changes
                v[32 * w + l].x += v[32 * w + l + o].x;
                v[32 * w + l].y += v[32 * w + l + o].y;
            }
    c2 r = v[0];
    for (int w = 1; w < NT / 32; ++w) r.x += v[32 * w].x, r.y += v[32 * w].y;
    return r;
}

static c2 final_sum(const std::vector<c2> &partial)
{
    std::vector<c2> acc(NT, c2{0, 0});
    for (size_t i = 0; i < partial.size(); ++i) acc[i % NT].x += partial[i].x, acc[i % NT].y += partial[i].y;
    return block_sum(acc);
}

static int run_freq(const std::string &cs, double C)
{
    size_t n = ((size_t)1 << 24) + 5;
    if (cs == "n3") n = 3;
    if (cs == "n2049") n = 2049;
    std::vector<c2> x(n);
    const size_t P0 = (n + 2047) / 2048, P = P0 < MAXP ? P0 : MAXP, stride = P * NT;
    if (cs == "chain") {  // thread 0's run: 1 + delta + delta + ..., each addition rounds up by about u64
        x.assign(n, c2{0, 0});
        x[0] = x[1] = c2{1, 0};
        for (size_t i = stride; i + 1 < n; i += stride) x[i] = c2{1, 0}, x[i + 1] = c2{0x1p-53 * (1 + 0x1p-10), 0};
    } else {
        for (auto &v : x) {
            const double a = uni() * TWO_PI, m = 0.5 + uni();
            v = c2{m * std::cos(a), m * std::sin(a)};
        }
    }
    std::vector<c2> partial(P);
    for (size_t b = 0; b < P; ++b) {
        std::vector<c2> acc(NT, c2{0, 0});
        for (int t = 0; t < NT; ++t)
            for (size_t i = b * NT + t; i + 1 < n; i += stride) {
                const c2 a = x[i + 1], bb = x[i];
                acc[t].x += std::fma(a.x, bb.x, a.y * bb.y);
                acc[t].y += std::fma(a.y, bb.x, -(a.x * bb.y));
            }
        partial[b] = block_sum(acc);
    }
    const c2 got = final_sum(partial);
    f128 sx = 0, sy = 0;
    double T = 0;
    for (size_t i = 0; i + 1 < n; ++i) {
        const c2 a = x[i + 1], bb = x[i];
        sx += (f128)a.x * bb.x + (f128)a.y * bb.y;
        sy += (f128)a.y * bb.x - (f128)a.x * bb.y;
        T += std::hypot(a.x, a.y) * std::hypot(bb.x, bb.y);
    }
    const size_t m = (n - 1 + stride - 1) / stride;
    const double D = 2 + m + 5 + 7 + (P + NT - 1) / NT + 5 + 7;
    const double err = std::hypot((double)((f128)got.x - sx), (double)((f128)got.y - sy));
    printf("{\"kernel\": \"freq\", \"case\": \"%s\", \"n\": %zu, \"worst\": %.6g, \"depth\": %g}\n", cs.c_str(), n,
           err / (C * U64 * D * T), D);
    return 0;
}

static c2 cmul64(c2 a, c2 b)  // a.x*b.x - a.y*b.y, a.x*b.y + a.y*b.x as nvcc contracts them
{
    return c2{std::fma(a.x, b.x, -(a.y * b.y)), std::fma(a.x, b.y, a.y * b.x)};
}

static int run_timing(unsigned N, unsigned D, size_t n, const std::string &cs, double C)
{
    const double alpha = 0.5, pi = 3.14159265358979323846;
    const unsigned ntaps = 2 * N * D + 1, ntaps4 = (ntaps + 3) & ~3u, nd = N * D;
    std::vector<double> h(ntaps4, 0.0);
    const int dd = (int)std::floor((double)ntaps / 2.0);
    for (unsigned i = 0; i < ntaps; ++i) {  // cb_qfilt_taps_f64
        const double tt = (double)((int)i - dd) / (double)N, two = 2.0 * alpha * tt;
        h[i] = std::fabs(two) == 1.0 ? std::sin(pi * alpha * tt) / (8.0 * tt)
                                     : (alpha * std::cos(pi * alpha * tt)) / (pi * (1.0 - two * two));
    }
    std::vector<c2> x(n), qin(n), din(n);
    std::vector<long double> cl(n), sl(n);
    for (size_t m = 0; m < n; ++m) {
        if (cs == "noise") {
            x[m] = c2{uni() * 2 - 1, uni() * 2 - 1};
        } else {  // QPSK symbols held for N samples
            const uint64_t r = next_u64();
            x[m] = m % N == 0 ? c2{(r & 1) ? 1.0 : -1.0, (r & 2) ? 1.0 : -1.0} : x[m - 1];
        }
        const double arg = -pi * (double)m / (double)N;
        const c2 r = c2{std::cos(arg), std::sin(arg)};
        cl[m] = cosl((long double)arg);
        sl[m] = sinl((long double)arg);
        qin[m] = cmul64(c2{x[m].x, -x[m].y}, r);
        din[m] = cmul64(x[m], r);
    }
    const size_t ntiles = (n + 1023) / 1024, P0 = ntiles, P = P0 < MAXP ? P0 : MAXP;
    std::vector<c2> partial(P);
    for (size_t b = 0; b < P; ++b) {
        std::vector<c2> acc(NT, c2{0, 0});
        for (size_t tile = b; tile < ntiles; tile += P)
            for (int t = 0; t < NT; ++t)
                for (int u = 0; u < 4; ++u) {
                    const long long i = (long long)tile * 1024 + 4 * t + u, m = i - (long long)nd;
                    if (i >= (long long)n || m < 0) continue;
                    c2 y{0, 0};
                    for (unsigned k = 0; k < ntaps4; ++k) {  // the register window's FMA chain, taps in order
                        const long long e = i - (long long)k;
                        const c2 q = e >= 0 ? qin[e] : c2{0, 0};
                        y.x = std::fma(h[k], q.x, y.x);
                        y.y = std::fma(h[k], q.y, y.y);
                    }
                    const c2 p = cmul64(y, din[m]);
                    acc[t].x += p.x;
                    acc[t].y += p.y;
                }
        partial[b] = block_sum(acc);
    }
    const c2 got = final_sum(partial);
    // reference: long double throughout, r from the same f64 argument
    long double sx = 0, sy = 0;
    double W = 0;
    for (size_t i = nd; i < n; ++i) {
        long double yx = 0, yy = 0, A = 0;
        for (unsigned k = 0; k < ntaps && k <= i; ++k) {
            const size_t e = i - k;
            const long double qx = x[e].x * cl[e] + x[e].y * sl[e], qy = x[e].x * sl[e] - x[e].y * cl[e];
            yx += h[k] * qx;
            yy += h[k] * qy;
            A += std::fabs(h[k]) * std::hypot(x[e].x, x[e].y);
        }
        const size_t m = i - nd;
        const long double dx = x[m].x * cl[m] - x[m].y * sl[m], dy = x[m].x * sl[m] + x[m].y * cl[m];
        sx += yx * dx - yy * dy;
        sy += yx * dy + yy * dx;
        W += std::hypot(x[m].x, x[m].y) * A;
    }
    const size_t tiles_per = (ntiles + P - 1) / P;
    const double Dt = 2 + 4 * tiles_per + 5 + 7 + (P + NT - 1) / NT + 5 + 7;
    const double err = std::hypot((double)(got.x - sx), (double)(got.y - sy));
    printf("{\"kernel\": \"timing\", \"case\": \"%s\", \"N\": %u, \"D\": %u, \"n\": %zu, \"worst\": %.6g}\n", cs.c_str(),
           N, D, n, err / (C * U64 * (ntaps4 + Dt) * W));
    return 0;
}

int main(int argc, char **argv)
{
    if (argc >= 6 && !strcmp(argv[1], "nco")) return run_nco(argv[2], argv[3], atof(argv[4]), atof(argv[5]));
    if (argc >= 4 && !strcmp(argv[1], "freq")) return run_freq(argv[2], atof(argv[3]));
    if (argc >= 7 && !strcmp(argv[1], "timing"))
        return run_timing((unsigned)atoi(argv[2]), (unsigned)atoi(argv[3]), (size_t)atoll(argv[4]), argv[5], atof(argv[6]));
    fprintf(stderr, "usage: phase_emul nco <old|fixed> <case> A B | freq <case> C | timing N D n <case> C\n");
    return 2;
}
