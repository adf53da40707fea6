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
