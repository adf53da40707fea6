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
