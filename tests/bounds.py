"""Float64 references and per-output error bounds (NumPy only, no GPU).

A FIR output y_n = sum_k h_k x_{n-k} computed in f32 carries an error relative to the terms that form it, not to the
frame's norm: the bound checked here is, for EVERY output,

    |got_n - exact_n| <= tol * A_n,    A_n = sum_k |h_k| |x_{n-k}|,

with exact_n the complex128 direct convolution.  Relative L2 over a frame or a 64-sample window cannot see one wrong
output among loud neighbours, nor a quiet output that is wrong by 1e-3 of itself; this can.

The FM discriminator theta_n = arg(y_n conj(y_{n-1})) inherits it: an error of tol * A_n in y_n turns the angle by at
most about tol * A_n / |y_n|, so modulo 2 pi

    |got_n - theta_n| <= tol * (A_n / |y_n| + A_{n-1} / |y_{n-1}|) + EPS_ATAN.

Outputs whose bound exceeds pi say nothing (y_n is cancellation noise) and are the only ones skipped.
"""
import numpy as np

# Absolute error of fm_angle_fast (misc_kernels.cuh: odd degree-17 polynomial of min/max, quadrant from the sign bits)
# against the exact angle of the same f32 product, measured on the CPU with the NumPy port `fm_angle_fast_np` below
# over 2^22 random products and along the octant edges: 2.8e-7 rad, most of it the f32 rounding of results near pi.  Rounded
# up with margin.
EPS_ATAN = 4e-7


def _stream(x, taps, state, interp):
    """(taps used, history ++ zero-stuffed x in chronological order, number of history samples)"""
    t = np.asarray(taps, np.complex128)
    st = np.zeros(len(t), np.complex128) if state is None else np.asarray(state, np.complex128)
    t = t[: min(len(t), len(st))]
    x = np.asarray(x, np.complex128)
    L = max(int(interp), 1)
    xs = np.zeros(len(x) * L, np.complex128)
    xs[::L] = x
    return t, np.concatenate([st[::-1], xs]), len(st)


def fir64(x, taps, state=None, interp=1, decim=1):
    """The product's FIR in complex128: zero-stuff by `interp` first, filter with the newest-first `state` as the
    samples before x (None: zeros of the taps' length; taps beyond the state's length unused), keep outputs
    0, D, 2D.. of this call.  Direct convolution on purpose: an FFT convolution's error is relative to the frame and
    would hide the quiet outputs.  Returns (y, state after the call)."""
    t, full, h = _stream(x, taps, state, interp)
    n = len(full) - h
    with np.errstate(all="ignore"):
        y = np.convolve(full, t)[h : h + n] if len(t) else np.zeros(n, np.complex128)
    return y[:: max(int(decim), 1)], full[::-1][:h].copy()


def fir_mag64(x, taps, state=None, interp=1, decim=1):
    """A_n = sum_k |h_k| |x_{n-k}|: the same operation on magnitudes (float64)"""
    t, full, h = _stream(x, taps, state, interp)
    n = len(full) - h
    with np.errstate(all="ignore"):
        a = np.convolve(np.abs(full), np.abs(t))[h : h + n] if len(t) else np.zeros(n)
    return a[:: max(int(decim), 1)]


def mix64(x, dphase, phase=0.0):
    """Mixer in float64 with the product's phase law: y_n = x_n exp(j (phase + n dphase)), dphase wrapped into
    [0, 2 pi), phase carried.  Returns (y, phase after the call)."""
    x = np.asarray(x, np.complex128)
    d = float(np.mod(dphase, 2 * np.pi))
    ph = phase + np.arange(len(x)) * d
    return x * np.exp(1j * ph), float(np.mod(phase + len(x) * d, 2 * np.pi))


def fm64(y, prev=0j):
    """FM discriminator in float64: arg(y_n conj(y_{n-1})), y_{-1} = prev"""
    y = np.asarray(y, np.complex128)
    p = np.concatenate([[complex(prev)], y[:-1]])
    return np.angle(y * np.conj(p))


def fir_bound_report(got, exact, A, tol=1e-5, idx=None):
    """(number of failing outputs, worst index, worst ratio |err| / (tol A)) over every output, or over the outputs
    `idx` only; see assert_fir_bound"""
    g = np.asarray(got).astype(np.complex128).ravel()
    e = np.asarray(exact, np.complex128).ravel()
    a = np.asarray(A, np.float64).ravel()
    assert g.shape == e.shape == a.shape, (g.shape, e.shape, a.shape)
    fin = np.isfinite(e.real) & np.isfinite(e.imag)
    bad = np.zeros(len(g), bool)
    # non-finite exact values: the non-finite pattern (per component) must match exactly
    bad |= ~fin & ((np.isfinite(g.real) != np.isfinite(e.real)) | (np.isfinite(g.imag) != np.isfinite(e.imag)))
    with np.errstate(all="ignore"):
        err = np.abs(g - e)
        ratio = np.where(fin, err / (tol * np.where(a > 0, a, 1.0)), 0.0)
    ratio = np.where(fin & (a == 0), np.where(g == 0, 0.0, np.inf), ratio)  # A_n = 0: exactly 0
    ratio = np.where(fin & ~np.isfinite(err), np.inf, ratio)
    bad |= ratio > 1.0
    r = np.where(bad & ~fin, np.inf, ratio)
    if idx is not None:
        keep = np.zeros(len(r), bool)
        keep[np.asarray(idx, np.int64)] = True
        bad &= keep
        r = np.where(keep, r, 0.0)
    nbad = int(bad.sum())
    worst = int(np.argmax(r)) if len(r) else 0
    return nbad, worst, float(r[worst]) if len(r) else 0.0


def assert_fir_bound(got, exact, A, tol=1e-5, what="", idx=None):
    """|got_n - exact_n| <= tol A_n for every n (or every n in idx); A_n == 0 -> got_n == 0; non-finite exact -> the
    same non-finite pattern"""
    nbad, worst, ratio = fir_bound_report(got, exact, A, tol, idx)
    assert nbad == 0, (f"{what}: {nbad} of {np.size(exact)} outputs outside tol*A (tol {tol:g}); worst index {worst}, "
                       f"|err|/(tol*A) = {ratio:.3g}, got {np.ravel(got)[worst]}, exact {np.ravel(exact)[worst]}, "
                       f"A {np.ravel(A)[worst]:.3g}")


def fm_bound_report(got, y_exact, A, tol=1e-5, y_prev=0j, A_prev=0.0, idx=None):
    """(failing outputs, worst index, worst ratio, skipped outputs) of the FM bound over every output, or over the
    outputs `idx` only; see assert_fm_bound"""
    g = np.asarray(got, np.float64).ravel()
    y = np.asarray(y_exact, np.complex128).ravel()
    a = np.asarray(A, np.float64).ravel()
    assert g.shape == y.shape == a.shape, (g.shape, y.shape, a.shape)
    th = fm64(y, y_prev)
    with np.errstate(all="ignore"):
        # y_n = 0 (A_n = 0 included: the angle of an exact zero is a convention of signed zeros) conditions nothing
        c = np.where(np.abs(y) > 0, a / np.where(np.abs(y) > 0, np.abs(y), 1.0), np.inf)
        cp = np.concatenate([[A_prev / abs(y_prev) if y_prev != 0 else np.inf], c[:-1]])
        bound = tol * (c + cp) + EPS_ATAN
        d = np.abs(g - th) % (2 * np.pi)
        d = np.minimum(d, 2 * np.pi - d)
    ok = ~(bound <= np.pi)  # ill-conditioned (or undefined) outputs are skipped
    ok |= d <= bound
    with np.errstate(all="ignore"):
        r = np.where(bound <= np.pi, d / bound, 0.0)
    if idx is not None:
        keep = np.zeros(len(r), bool)
        keep[np.asarray(idx, np.int64)] = True
        ok |= ~keep
        r = np.where(keep, r, 0.0)
    nbad = int((~ok).sum())
    worst = int(np.argmax(r)) if len(r) else 0
    return nbad, worst, float(r[worst]) if len(r) else 0.0, int((~(bound <= np.pi)).sum())


def assert_fm_bound(got, y_exact, A, tol=1e-5, what="", y_prev=0j, A_prev=0.0, idx=None):
    """every FM output (or every one in idx) within tol (A_n/|y_n| + A_{n-1}/|y_{n-1}|) + EPS_ATAN of the float64
    angle (modulo 2 pi), y_{-1} = y_prev (0: the stream's first output is skipped)"""
    nbad, worst, ratio, skipped = fm_bound_report(got, y_exact, A, tol, y_prev, A_prev, idx)
    assert nbad == 0, (f"{what}: {nbad} of {np.size(got)} FM outputs outside the bound ({skipped} ill-conditioned "
                       f"skipped); worst index {worst}, |err|/bound = {ratio:.3g}")


def fm_angle_fast_np(s, p):
    """NumPy port of fm_angle_fast (misc_kernels.cuh) in f32, without FMA contraction (one more rounding per step:
    an upper estimate of the device's rounding error)"""
    f = np.float32
    s = np.asarray(s, np.complex64)
    p = np.asarray(p, np.complex64)
    br, bi = p.real, -p.imag
    tr = s.real * br - s.imag * bi
    ti = s.real * bi + s.imag * br
    ax, ay = np.abs(tr), np.abs(ti)
    mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
    with np.errstate(all="ignore"):
        a = np.where(mx > 0, mn / np.where(mx > 0, mx, f(1)), f(0)).astype(np.float32)
    z = a * a
    q = np.full_like(z, f(0.0028340641874819994))
    for c in (-0.016005029901862144, 0.042587608098983765, -0.07495445758104324, 0.10636754333972931,
              -0.14202570915222168, 0.19992484152317047, -0.3333306610584259, 1.0):
        q = q * z + f(c)
    r = a * q
    r = np.where(ay > ax, f(1.57079632679489662) - r, r)
    r = np.where(np.signbit(tr), f(3.14159265358979324) - r, r)
    r = np.where(np.signbit(ti), -r, r).astype(np.float32)
    return r, tr, ti


def parity_sparse(taps):
    """True when the taps' non-zero entries leave some output without an aligned pair (x_{2j}, x_{2j+1}) of samples:
    no two adjacent non-zero taps ending at an even offset, or none ending at an odd offset (1 tap, every other tap
    zero, 2 taps...).  Such filters need the tensor-core kernels' per-sample quiet test."""
    nz = np.abs(np.asarray(taps)) != 0
    adj = nz[1:] & nz[:-1]  # adj[i]: taps i and i + 1 both non-zero, the pair ends at offset i + 1
    return bool(nz.any()) and not (adj[1::2].any() and adj[0::2].any())


# ---------------------------------------------------------------------------------------------------------------- FFT
# Every bin X_k = sum_n x_n W^{kn} is a sum over all inputs with unit-modulus twiddles, so its rounding error scales
# with S_f = sum_n |x_n| of its frame, not with |X_k| nor with the frame's norm.  Checked, for EVERY bin of EVERY
# frame of an N-point transform computed in f32 (u = 2^-24):
#
#     |got_k - X_k| <= tau * S_f + FFT_FLOOR * N * 2^-149      and      ||got_f - X_f||_2 <= rho ||X_f||_2 (+ floor)
#
#   power-of-two sizes (radix 16 passes, two-step splits):  tau = C_TAU log2(N) u,  rho = C_RHO log2(N) u
#   direct O(N^2) sum (N <= 128 otherwise):                  tau = rho = C_DIRECT u, whatever N
#   chirp-z (any other N, M = padded power of two):           tau = C_CHIRPZ log2(M) u,  rho = C_CHIRPZ_RHO log2(M) u
#
# with X the complex128 transform.  Exact cases: a frame with S_f = 0 gives exact zeros; a frame holding a non-finite
# input gives every bin non-finite (in at least one component), and every other frame of the batch stays finite and
# within its bounds.
#
# The constants are twice (at most) the worst ratio seen in the CPU emulation of the device arithmetic
# (tests/emul/fft2_emul.cpp; tests/test_fft_bounds_cpu.py checks them):
# - C_TAU: an impulse is the worst case, every output being a product of rounded twiddles.  The twiddle16 power tree
#   (depth 4), the bfly16 constant rotations and the table entries each add a rounding per 16-point digit: worst
#   emulated 2.05 (65536 points, 256 x 256 with twiddle16c), 1.88 (4096), 1.64 (256).
# - C_RHO: worst emulated 0.96 (a tone on an exact bin, 4096-point inverse); random frames 0.3 .. 0.53.  1.6 keeps
#   rho <= 2e-6 up to 2^20 points.
# - C_DIRECT: dft_direct_kernel multiplies by an exact-angle table entry (|dw| <= 0.71 u), rounds the complex
#   product (normwise <= 2 u |x_n| with the fused multiply-add, Jeannerod et al. 2017) and sums with Kahan
#   compensation (<= 2 u sum |terms| + O(N u^2) S_f = 2 u S_f): (0.71 + 2 + 2) u S_f, rounded up to 5 u S_f.
# - C_CHIRPZ, C_CHIRPZ_RHO: the emulation also runs the fused chirp-z kernel (bluestein_frames_kernel) on the same
#   passes, M = 512 .. 16384, with the chirp and its f32-rounded spectrum B exactly as bluestein_setup builds them.
#   It meets the S_f form with log2(M): worst 2.74 (impulses, N = 4095), norm 1.00 (random frames, N = 8191).  The
#   worst-case algebra would let the error grow with sqrt(N) (the inverse transform's input has sum |Z_k| ~
#   M sqrt(2N) |x|); neither this emulation nor a NumPy f32 emulation of the sequence up to M = 2^20 shows growth.
FFT_U = 2.0 ** -24
C_TAU = 4.0
C_RHO = 1.6
C_DIRECT = 5.0
C_CHIRPZ = 5.4
C_CHIRPZ_RHO = 2.0
FFT_FLOOR = 4.0  # absolute floor, in units of N * 2^-149 (chirp-z: M sqrt(2N) * 2^-149): subnormal frames


def chirpz_m(n):
    """padded size of the chirp-z plan: the least power of two >= max(256, 2N - 1) (bluestein_setup, api.cu)"""
    m = 256
    while m < 2 * n - 1:
        m <<= 1
    return m


def fft_path(n, direct=False):
    """the kind of plan cb_fft_create makes for N points: 'pow2' (2^3 .. 2^20), 'direct' (any other N <= 128, or up
    to 4096 with COMMS_B200_FFT_PATH=direct) or 'chirpz'"""
    if n >= 8 and n & (n - 1) == 0:
        return "pow2"
    return "direct" if n <= 128 or (direct and n <= 4096) else "chirpz"


def fft_constants(n, path):
    """(tau, rho, floor) of an N-point transform on `path`: |err_k| <= tau S_f + floor, ||err|| <= rho ||X|| +
    floor sqrt(N)"""
    if path == "direct":
        return C_DIRECT * FFT_U, C_DIRECT * FFT_U, FFT_FLOOR * n * 2.0 ** -149
    if path == "chirpz":
        m = chirpz_m(n)
        lm = np.log2(m)
        return C_CHIRPZ * lm * FFT_U, C_CHIRPZ_RHO * lm * FFT_U, FFT_FLOOR * m * np.sqrt(2 * n) * 2.0 ** -149
    assert path == "pow2", path
    return C_TAU * np.log2(n) * FFT_U, C_RHO * np.log2(n) * FFT_U, FFT_FLOOR * n * 2.0 ** -149


def fft64(x, n, inverse=False):
    """the product's unnormalised transform of every frame in complex128 (frames, n): X_k = sum x_n e^{-/+ 2 pi i kn/N}"""
    x = np.asarray(x).astype(np.complex128).reshape(-1, n)
    with np.errstate(all="ignore"):
        return np.fft.ifft(x, axis=1) * n if inverse else np.fft.fft(x, axis=1)


def fft_bound_report(got, x, n, inverse=False, path=None, exact=None):
    """Check every bin of every frame.  Returns (failures, worst bin ratio, worst norm ratio): failures is a list of
    messages naming the frame, the bin and the ratio; the ratios are over the finite frames with S_f > 0, as
    |err_k| / bin bound and ||err|| / norm bound (<= 1 passes).  `exact`: fft64(x, n, inverse) if already at hand."""
    path = path or fft_path(n)
    tau, rho, floor = fft_constants(n, path)
    x = np.asarray(x).reshape(-1, n)
    g = np.asarray(got).reshape(-1, n).astype(np.complex128)
    assert g.shape == x.shape, (g.shape, x.shape)
    X = fft64(x, n, inverse) if exact is None else np.asarray(exact).reshape(-1, n)
    xa = np.abs(x.astype(np.complex128))
    finite_in = np.isfinite(x.real).all(axis=1) & np.isfinite(x.imag).all(axis=1)
    with np.errstate(all="ignore"):
        S = xa.sum(axis=1)
        gfin = np.isfinite(g.real) & np.isfinite(g.imag)
        err = np.abs(g - X)
        bb = tau * S + floor
        rbin = err / bb[:, None]
        enorm = np.sqrt((err ** 2).sum(axis=1))
        nb = rho * np.sqrt((np.abs(X) ** 2).sum(axis=1)) + floor * np.sqrt(n)
        rnorm = enorm / nb
    fails, wbin, wnorm = [], 0.0, 0.0
    where = f"{path} N={n} {'inverse' if inverse else 'forward'}"
    for f in range(x.shape[0]):
        if not finite_in[f]:
            ok = ~gfin[f]
            if not ok.all():
                k = int(np.argmin(ok))
                fails.append(f"{where}: frame {f} holds a non-finite input but bin {k} is finite ({g[f, k]}); "
                             f"{int((~ok).sum())} of {n} bins finite")
            continue
        if not gfin[f].all():
            k = int(np.argmin(gfin[f]))
            fails.append(f"{where}: frame {f} (finite input) has non-finite bin {k} ({g[f, k]}); "
                         f"{int((~gfin[f]).sum())} of {n} bins non-finite")
            continue
        if S[f] == 0:
            if np.any(g[f] != 0):
                k = int(np.argmax(g[f] != 0))
                fails.append(f"{where}: frame {f} is all zeros but bin {k} is {g[f, k]} "
                             f"({int((g[f] != 0).sum())} of {n} bins non-zero)")
            continue
        k = int(np.argmax(rbin[f]))
        wbin, wnorm = max(wbin, float(rbin[f, k])), max(wnorm, float(rnorm[f]))
        if rbin[f, k] > 1:
            fails.append(f"{where}: frame {f} bin {k}: |err|/bound = {rbin[f, k]:.3g} ({int((rbin[f] > 1).sum())} of "
                         f"{n} bins outside), got {g[f, k]}, exact {X[f, k]}, bound {bb[f]:.3g}")
        if rnorm[f] > 1:
            fails.append(f"{where}: frame {f}: ||err||/(rho ||X||) = {rnorm[f]:.3g} (rho {rho:.3g})")
    return fails, wbin, wnorm


def assert_fft_bound(got, x, n, inverse=False, path=None, what="", exact=None):
    """every bin of every frame within its bound (see fft_bound_report); returns the worst (bin, norm) ratios"""
    fails, wbin, wnorm = fft_bound_report(got, x, n, inverse, path, exact)
    assert not fails, f"{what}: {len(fails)} failures; " + "; ".join(fails[:6])
    return wbin, wnorm


# ---------------------------------------------------------------------------------------------------- overlap-save FIR
OLS_N = 4096


def ols_bound(x, taps, hist=None):
    """Per-output bound of the overlap-save FIR (fir_ols_kernel, 4096-point frames, hop 4097 - K) for one call of
    x after the newest-first history `hist` (None: zeros): output n comes from frame f = n // hop, whose inputs are
    x_f = samples [f hop - (K - 1), f hop - (K - 1) + 4096) of the call (history before 0, zeros past the call's end).
    Forward transform, product with Hf and inverse each obey the FFT norm bound, so

        |err_n| <= (2 rho_4096 + u) ||H||_inf ||x_f||_2,   H = 4096-point DFT of the taps in float64 from the f32 taps.

    Returns (bound per output, frame index per output)."""
    t = np.asarray(taps, np.complex64).astype(np.complex128)
    K = len(t)
    hop = OLS_N - (K - 1)
    x = np.asarray(x).astype(np.complex128)
    h = np.zeros(K - 1, np.complex128) if hist is None else np.asarray(hist, np.complex128)[: K - 1][::-1]
    full = np.concatenate([np.zeros(K - 1 - len(h), np.complex128), h, x, np.zeros(OLS_N, np.complex128)])
    H = np.fft.fft(np.concatenate([t, np.zeros(OLS_N - K)]))
    frames = -(-len(x) // hop)
    win = np.lib.stride_tricks.sliding_window_view(np.abs(full), OLS_N)[::hop][:frames]  # index 0: sample -(K - 1)
    with np.errstate(all="ignore"):
        xn = np.sqrt((win ** 2).sum(axis=1))
    _, rho, _ = fft_constants(OLS_N, "pow2")
    f = np.arange(len(x)) // hop
    return (2 * rho + FFT_U) * np.abs(H).max() * xn[f], f


def ols_seams(n, ntaps):
    """first and last output of every overlap-save frame of an n-sample call"""
    hop = OLS_N - (ntaps - 1)
    s = np.arange(0, n, hop)
    return np.unique(np.clip(np.concatenate([s - 1, s]), 0, n - 1))


# ------------------------------------------------------------------------------------ phase laws: mixer, NCO, estimators
# References for the kernels whose output is a phase law (the stand-alone mixer, the NCO scan) and for the two f64
# estimators, with the per-output bounds that include/comms_b200.h states.  u32 = 2^-24, u64 = 2^-53.
#
# The exact phase is formed in double-double: k * dphase as a Dekker two-product, phase0 and the prefix of perr added
# with two-sums, and the result reduced against a three-part 2 pi (159 bits, from the integer below) with two-products
# for q * P1 and q * P2.  For |theta| < 2^33 the reduced phase is correct to about 2^-72 rad; it is then handed to
# long double (64-bit mantissa: 2^-64 pi) for sin and cos.  np.longdouble is NOT used for the reduction: its 64-bit
# 2 pi would be off by about 1e-10 rad at k * dphase ~ 2^32.
U32 = 2.0 ** -24
U64 = 2.0 ** -53
TWO_PI_2_200 = 10096689509235987743946820282484873672429286842977325943070736  # floor(2 pi 2^200)


def _two_pi_parts():
    from fractions import Fraction
    t = Fraction(TWO_PI_2_200, 1 << 200)
    p1 = float(t)
    p2 = float(t - Fraction(p1))
    p3 = float(t - Fraction(p1) - Fraction(p2))
    return p1, p2, p3


TWO_PI_P1, TWO_PI_P2, TWO_PI_P3 = _two_pi_parts()


def two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _split(a):
    c = 134217729.0 * a  # 2^27 + 1
    hi = c - (c - a)
    return hi, a - hi


def two_prod(a, b):
    """(p, e) with p + e = a * b exactly (Dekker; NumPy does not contract to FMA)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def dd_add(ah, al, bh, bl):
    s, e = two_sum(ah, bh)
    e = e + (al + bl)
    return two_sum(s, e)


def phase_exact(phase0, dphase, k, prefix=None):
    """theta = phase0 + k dphase + prefix reduced mod 2 pi into about [-pi, pi], as a double-double (hi, lo).
    k: integer array (k < 2^29); prefix: None, an array of doubles, or a (hi, lo) pair of arrays (exact sums)."""
    with np.errstate(all="ignore"):
        k = np.asarray(k, np.float64)
        h, l = two_prod(k, np.float64(dphase))
        h, l = dd_add(h, l, np.float64(phase0), 0.0)
        if prefix is not None:
            ph, pl = prefix if isinstance(prefix, tuple) else (np.asarray(prefix, np.float64), 0.0)
            h, l = dd_add(h, l, ph, pl)
        q = np.rint(h / TWO_PI_P1)
        q = np.where(np.isfinite(q), q, 0.0)
        a, b = two_prod(q, TWO_PI_P1)
        h, l = dd_add(h, l, -a, -b)
        a, b = two_prod(q, TWO_PI_P2)
        h, l = dd_add(h, l, -a, -b)
        h, l = dd_add(h, l, -q * TWO_PI_P3, 0.0)
    return h, l


def _cis_ld(h, l):
    """(cos, sin) of the double-double phase, in long double"""
    t = np.asarray(h).astype(np.longdouble) + np.asarray(l).astype(np.longdouble)
    return np.cos(t), np.sin(t)


def _err_ld(got, c, s):
    """|got - (c + j s)| with the reference kept in long double"""
    g = np.asarray(got).astype(np.complex128)
    with np.errstate(all="ignore"):
        dr = g.real.astype(np.longdouble) - c
        di = g.imag.astype(np.longdouble) - s
        return np.sqrt(dr * dr + di * di).astype(np.float64)


# ---- mixer: y_n = x_n e^{j theta_n}, theta_n = phase + n dphase, carried across calls
# The f64 part (fma(i, dphase, phase0) and the Cody-Waite reduction) rounds once at |theta|: u64 (|phase0| + n dphase)
# rad.  The f32 part rests on sincosf's documented maximum error of 2 ulp (CUDA programming guide, Table of
# single-precision functions), so it is derived rather than emulated: per component 2 u32 (sincosf) + u32 (the fmaf of
# the hi/lo correction) + the second-order term lo^2/2 < 2^-47, i.e. |r - e^{j theta}| <= 3 sqrt(2) u32 for one
# rotation; the vector path's r_k = r0 s_k adds a second rotation and a fused complex product (2 u32, Jeannerod et al.
# 2017); the final x r adds 2 u32 |x|: 2 (3 sqrt 2) + 2 + 2 = 12.5, rounded up to C_MIX = 13.  Subnormal outputs add
# an absolute floor of 2^-148 (two roundings at 2^-150 per component).  The carried phase (advance_phase, api.cu)
# rounds once to f64 per call (u64 2 pi) after a long double fmodl whose 2 pi is off by 2 pi 2^-64 per turn.
C_MIX = 13.0
MIX_FLOOR = 2.0 ** -148


def mix_exact(x, dphase, phase0, start=0):
    """(cos, sin) of the exact phase for the samples start .. start + len(x) of a stream whose sample 0 had phase
    phase0 (dphase as the handle holds it), and the exact x e^{j theta} in long double (re, im)"""
    k = start + np.arange(len(x), dtype=np.int64)
    c, s = _cis_ld(*phase_exact(phase0, dphase, k))
    xr = np.asarray(x).real.astype(np.longdouble)
    xi = np.asarray(x).imag.astype(np.longdouble)
    return xr * c - xi * s, xr * s + xi * c


def mix_carry(phase_in, m, dphase):
    """what one call of m samples adds to the `carried` term: the f64 rounding of the carried phase (2 pi) and the long
    double steps of advance_phase (2^-64 (|phase_in| + m dphase) each, with a 64-bit 2 pi), in units of u64"""
    return 2 * np.pi + 2.0 ** -9 * (abs(phase_in) + m * dphase)


def mix_bound(x, dphase, phase0, start=0, carried=0.0):
    """per-output bound (C_MIX u32 + u64 (|phase0| + n dphase + 8 pi + carried)) |x_n| + MIX_FLOOR, n counted from the
    stream's start; 8 pi covers the rounding of 2 dphase, 3 dphase and the quad's first phase; `carried`: the sum of
    mix_carry over the calls before this one"""
    n = start + np.arange(len(x), dtype=np.float64)
    return (C_MIX * U32 + U64 * (abs(phase0) + n * dphase + 8 * np.pi + carried)) * np.abs(
        np.asarray(x).astype(np.complex128)) + MIX_FLOOR


def mix_bound_report(got, x, dphase, phase0, start=0, carried=0.0, idx=None):
    """(failures, worst index, worst ratio): every output within mix_bound; a zero input gives an exact zero; a
    non-finite input gives a non-finite output (in at least one component); finite inputs give finite outputs"""
    g = np.asarray(got).astype(np.complex128)
    x = np.asarray(x).astype(np.complex128)
    fin_x = np.isfinite(x.real) & np.isfinite(x.imag)
    xs = np.where(fin_x, x, 0)
    er, ei = mix_exact(xs, dphase, phase0, start)
    with np.errstate(all="ignore"):
        dr = g.real.astype(np.longdouble) - er
        di = g.imag.astype(np.longdouble) - ei
        err = np.sqrt(dr * dr + di * di).astype(np.float64)
        r = err / mix_bound(xs, dphase, phase0, start, carried)
    fin_g = np.isfinite(g.real) & np.isfinite(g.imag)
    r = np.where(fin_x, np.where(fin_g, r, np.inf), np.where(fin_g, np.inf, 0.0))
    r = np.where(fin_x & (x == 0), np.where(g == 0, 0.0, np.inf), r)
    if idx is not None:
        keep = np.zeros(len(r), bool)
        keep[np.asarray(idx, np.int64)] = True
        r = np.where(keep, r, 0.0)
    bad = np.nonzero(r > 1)[0]
    w = int(np.argmax(r)) if len(r) else 0
    fails = [f"mixer output {int(bad[0]) + start} (stream index): |err|/bound = {r[bad[0]]:.3g}, got {g[bad[0]]}, "
             f"x {x[bad[0]]}; {len(bad)} outputs outside"] if len(bad) else []
    return fails, w, float(r[w]) if len(r) else 0.0


# ---- NCO: out_k = e^{j phi_k}, phi_k = phase_0 + (k + 1) dphase + sum_{i <= k} perr_i (mod 2 pi), carried
# Causal bound (only perr[0..k] enters the bound of output k):
#
#     |out_k - e^{j phi_k}| <= u64 (C_NCO_A (|phase_0| + 2 pi (1 + calls_k + chunks_k)) + C_NCO_B S_k + C_SINCOS)
#
# S_k = sum_{i <= k} |perr_i| over the stream, calls_k = calls before the one holding k (each re-reduces the carried
# phase), chunks_k = scan chunks of 2^21 samples before k in its call (each re-reduces the carry).  C_NCO_A and
# C_NCO_B are twice (at most) the worst ratios of the CPU emulation of the device's f64 operation sequence
# (tests/emul/phase_emul.cpp, checked in tests/test_phase_bounds_cpu.py): 0.52 of the bound with phase_0 = 1e6 + 0.3
# (ph0 + reduce(...) + (off + v) rounds twice at |phase_0|), 0.56 with perr = 1 at each thread's first sample and 2^-53 (1 + 2^-20) elsewhere
# (every addition of the thread, warp and CTA scans rounds the same way), 0.11 on random perr over three scan chunks.
# C_SINCOS: the device's f64 sincos is within 2 ulp per component (CUDA programming guide): 2 ulp(1) sqrt 2 = 4 sqrt
# 2 u64, rounded up to 6.  A non-finite perr_j makes out_j.., and the carried phase, NaN; out_0 .. out_{j-1} stay
# within the bound.
C_NCO_A = 2.0
C_NCO_B = 16.0
C_SINCOS = 6.0
NCO_CHUNK = 1024 * 2048


def exact_prefix(perr):
    """Inclusive prefix sums of perr as double-double arrays (hi, lo), exact to about 2^-100 of their size.  Entries
    on the dyadic grid int * 2^-40 (|int| < 2^30) are summed exactly in int64; the others (at most a few thousand:
    huge values, subnormals, mixed magnitudes) are summed exactly with Fraction and added in double-double.
    Non-finite entries give NaN from their index on."""
    from fractions import Fraction
    p = np.asarray(perr, np.float64)
    fin = np.isfinite(p)
    s = np.where(fin, p, 0.0) * 2.0 ** 40
    grid = fin & (s == np.rint(s)) & (np.abs(s) < 2.0 ** 30)
    ints = np.where(grid, s, 0.0).astype(np.int64)
    hi = np.cumsum(ints).astype(np.float64) * 2.0 ** -40  # |cumsum| < 2^53: exact
    lo = np.zeros_like(hi)
    off = np.nonzero(fin & ~grid)[0]
    assert len(off) <= 8192, "exact_prefix: too many off-grid entries"
    if len(off):
        acc = Fraction(0)
        bounds = list(off) + [len(p)]
        for j, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
            acc += Fraction(float(p[a]))
            ah = float(acc)
            al = float(acc - Fraction(ah))
            h2, l2 = dd_add(hi[a:b], lo[a:b], ah, al)
            hi[a:b], lo[a:b] = h2, l2
    bad = np.nonzero(~fin)[0]
    if len(bad):
        hi[bad[0]:] = np.nan
        lo[bad[0]:] = np.nan
    return hi, lo


def nco_exact(phase0, dphase, perr, start=0, prefix=None):
    """(cos, sin) in long double of e^{j phi_k} for the outputs k = start .. start + len(perr) - 1 of a stream whose
    phase was phase0 before its output 0; `prefix`: exact (hi, lo) prefix sums of the stream's perr at these outputs
    (default: of perr alone, i.e. start == 0 or no earlier perr)"""
    pre = exact_prefix(perr) if prefix is None else prefix
    k = start + 1 + np.arange(len(perr), dtype=np.int64)
    return _cis_ld(*phase_exact(phase0, dphase, k, pre))


def nco_bound(phase0, S, calls=0, chunks=0):
    return U64 * (C_NCO_A * (abs(phase0) + 2 * np.pi * (1 + calls + np.asarray(chunks))) + C_NCO_B * np.asarray(S)
                  + C_SINCOS)


def nco_bound_report(got, c, s, bound, nonfinite_from=None):
    """(failures, worst index, worst ratio) of NCO outputs against (c + j s) and the per-output bound; from index
    `nonfinite_from` on every output must be NaN (in both components)"""
    g = np.asarray(got).astype(np.complex128)
    n = len(g)
    j = n if nonfinite_from is None else int(nonfinite_from)
    err = _err_ld(g[:j], c[:j], s[:j])
    with np.errstate(all="ignore"):
        r = np.where(np.isfinite(err), err / np.asarray(bound)[:j], np.inf)
    fails = []
    bad = np.nonzero(~(r <= 1))[0]
    if len(bad):
        b = int(bad[0])
        fails.append(f"NCO output {b}: |err|/bound = {r[b]:.3g} (|err| {err[b]:.3g}, bound {np.asarray(bound)[b]:.3g}); "
                     f"{len(bad)} of {j} causal outputs outside")
    if j < n:
        nn = ~(np.isnan(g[j:].real) & np.isnan(g[j:].imag))
        if nn.any():
            fails.append(f"NCO output {j + int(np.argmax(nn))} at or after the non-finite perr[{j}] is not NaN "
                         f"({int(nn.sum())} of {n - j})")
    w = int(np.argmax(np.where(np.isfinite(r), r, np.inf))) if len(r) else 0
    return fails, w, float(r[w]) if len(r) else 0.0


# ---- f64 estimators: |est - arg S| <= asin(E / |S|) + EST_ABS
# Frequency estimator, S = sum_{i < n-1} x_{i+1} conj(x_i):  E = C_FREQ u64 D_F sum |x_{i+1}| |x_i|, where D_F counts
# the additions on one term's way to the result at the launch shape (P = min(ceil(n / 2048), 1184) CTAs of 256
# threads): the product (2), the thread's run of m = ceil((n-1) / (256 P)) terms, the warp tree (5) and the CTA's 7
# warp partials, the final CTA's ceil(P / 256) partials per thread, its warp tree and warp partials.  C_FREQ = sqrt 2
# (each of the real and imaginary sums obeys the first-order bound D_F u64 sum |t|; the complex error is at most
# sqrt 2 times that).  The emulation attains 0.45 of it with terms built so that one thread's additions all round the
# same way (random-phase input: 1.3e-5).  EST_ABS = 4 ulp(pi): atan2, the reference's own rounding of arg S and the
# roundings of -N arg / 2 pi.
C_FREQ = np.sqrt(2.0)
EST_ABS = 2.0 ** -49
EST_BLOCKS = 148 * 8


def freq_depth(n):
    p = min(-(-max(n, 1) // 2048), EST_BLOCKS)
    m = -(-(n - 1) // (256 * p))
    return 2 + m + 5 + 7 + -(-p // 256) + 5 + 7


def _dd_tree_sum(h, l):
    """double-double sum of the pairs (h_i, l_i) by a pairwise tree"""
    h, l = np.asarray(h, np.float64), np.asarray(l, np.float64)
    while len(h) > 1:
        if len(h) & 1:
            h, l = np.append(h, 0.0), np.append(l, 0.0)
        h, l = dd_add(h[0::2], l[0::2], h[1::2], l[1::2])
    return (float(h[0]), float(l[0])) if len(h) else (0.0, 0.0)


def freq_exact(x):
    """(S as complex128 rounded from its double-double, sum |x_{i+1}| |x_i|, S as ((re hi, re lo), (im hi, im lo)))"""
    x = np.asarray(x, np.complex128)
    a, b = x[1:], x[:-1]
    with np.errstate(all="ignore"):
        p1, e1 = two_prod(a.real, b.real)
        p2, e2 = two_prod(a.imag, b.imag)
        p3, e3 = two_prod(a.imag, b.real)
        p4, e4 = two_prod(a.real, b.imag)
        re = _dd_tree_sum(np.concatenate([p1, p2]), np.concatenate([e1, e2]))
        im = _dd_tree_sum(np.concatenate([p3, -p4]), np.concatenate([e3, -e4]))
        T = float(np.sum(np.abs(a) * np.abs(b)))
    return complex(re[0] + re[1], im[0] + im[1]), T, (re, im)


def angle_dd(re, im):
    """arg of the double-double complex number ((re hi, re lo), (im hi, im lo)), in long double"""
    return float(np.arctan2(np.longdouble(im[0]) + np.longdouble(im[1]), np.longdouble(re[0]) + np.longdouble(re[1])))


def est_bound_report(est, S_abs, E, arg_exact, scale=1.0, what=""):
    """(ok, ratio, skipped): |est - arg_exact| (mod 2 pi, times `scale` for the timing estimator) within
    scale (asin(E / |S|) + EST_ABS); skipped when E >= |S| (the estimate must still be finite)"""
    if not (E < S_abs):
        return bool(np.isfinite(est)), 0.0, True
    d = abs(est - arg_exact * scale) / abs(scale)
    d = min(d % (2 * np.pi), 2 * np.pi - d % (2 * np.pi))
    b = np.arcsin(E / S_abs) * (1 + 1e-9) + EST_ABS
    return d <= b, d / b, False


# Timing estimator: S = sum_i qout_i dout_i, qout = q * qin (2ND+1 real taps), qin_m = conj(x_m) r_m, dout_i =
# x_{i-ND} r_{i-ND}, r_m = e^{-j fl(fl(-pi m) / N)} (the reference's operation order).
#   E = u64 (C_TIM (ntaps4 + D_T) + 2 (C_SINCOS + 2)) sum_i |dout_i| A_i,   A_i = sum_k |q_k| |qin_{i-k}|
# ntaps4 = the FMA chain of the register window (taps padded to four), D_T the partial sums at the launch shape (the
# product, each thread's 4 outputs per tile over its tiles, the CTA and final trees as for the frequency estimator),
# 2 (C_SINCOS + 2) the device sincos and the products qin = conj(x) r, din = x r, which scale both factors.  C_TIM =
# sqrt 2 as above.  This one is a worst-case first-order bound, not a calibrated one: the emulation's worst ratio on
# noise and QPSK input is 2.7e-3 (no input was found that aligns the roundings of the 4-tap-group FMA chain).  The timing estimate is -N arg(S) / 2 pi, so its bound is (N / 2 pi) (asin(E / |S|) + EST_ABS).
C_TIM = np.sqrt(2.0)


def timing_depth(n, ntaps):
    p = min(-(-max(n, 1) // 1024), EST_BLOCKS)
    tiles = -(-(-(-n // 1024)) // p)
    return 2 + 4 * tiles + 5 + 7 + -(-p // 256) + 5 + 7


def timing_taps(n, d, alpha):
    """the f64 taps the library uses: cb_qfilt_taps_f64(2 n d + 1, alpha, n), recomputed here"""
    real_n = 2 * n * d + 1
    dd = int(np.floor(real_n / 2.0))
    t = np.empty(real_n)
    for i in range(real_n):
        tt = float(i - dd) / float(n)
        two = 2.0 * alpha * tt
        if abs(two) == 1.0:
            t[i] = np.sin(np.pi * alpha * tt) / (8.0 * tt)
        else:
            t[i] = (alpha * np.cos(np.pi * alpha * tt)) / (np.pi * (1.0 - two * two))
    return t


def timing_exact(x, taps, N, D):
    """(running S_i = sum_{i' <= i} qout_i' dout_i' as complex long double per i, running W_i = sum |dout| A, per
    i): the exact sums of every prefix length of x, so that one call serves every n.  qout in long double by direct
    convolution (error <= ntaps 2^-64 A_i), r from the reference's f64 argument with long double sin and cos."""
    x = np.asarray(x, np.complex128)
    n = len(x)
    m = np.arange(n, dtype=np.float64)
    arg = (-np.pi * m) / float(N)  # the f64 argument, bit for bit (pi * m first, then / N)
    c, s = np.cos(arg.astype(np.longdouble)), np.sin(arg.astype(np.longdouble))
    xr, xi = x.real.astype(np.longdouble), x.imag.astype(np.longdouble)
    qin = (xr * c + xi * s) + 1j * (xr * s - xi * c)  # conj(x) r
    din = (xr * c - xi * s) + 1j * (xr * s + xi * c)  # x r
    t = np.asarray(taps).astype(np.longdouble)
    qout = np.convolve(qin.astype(np.clongdouble), t)[:n]
    A = np.convolve(np.abs(qin).astype(np.longdouble), np.abs(t))[:n]
    nd = N * D
    dout = np.zeros(n, np.clongdouble)
    dout[nd:] = din[: n - nd] if nd < n else []
    S = np.cumsum(qout * dout)
    W = np.cumsum((np.abs(dout) * A).astype(np.float64))
    return S, W


def timing_E(n, ntaps, W):
    ntaps4 = (ntaps + 3) & ~3
    return U64 * (C_TIM * (ntaps4 + timing_depth(n, ntaps)) + 2 * (C_SINCOS + 2)) * W * (1 + 1e-6)
