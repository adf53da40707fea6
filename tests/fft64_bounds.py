"""Error bounds of the Complex<f64> FFT (cb_fft_f64, include/comms_b200.h), its exact reference and the ctypes wrapper
of its CPU emulation (tests/emul/fft_f64_emul.cpp), shared by tests/test_fft_f64_cpu.py and tests/test_gpu_fft_f64.py."""
import math
import os

import numpy as np

U64 = 2.0 ** -53
TINY = 2.0 ** -1074

# the plan's paths (the emulation returns the same codes)
DIRECT, FRAMES, TWOSTEP, CHIRPZ = 0, 1, 2, 3
FRAME_MAX = 4096
DIRECT_MAX = 128
# scipy.fft over clongdouble against the exact transform: <= 1.1e-19 S_f measured at N = 64 .. 4096 against a direct
# long-double DFT (about 1e-3 of u S_f); counted into every check with a factor 8 of margin
REF_TAU = 1e-18


def path_of(n):
    pow2 = n & (n - 1) == 0
    if pow2 and n >= 8:
        return FRAMES if n <= FRAME_MAX else TWOSTEP
    if pow2 or n <= DIRECT_MAX:
        return DIRECT
    return CHIRPZ


def chirp_m(n):
    m = 8
    while m < 2 * n - 1:
        m *= 2
    return m


def constants(n):
    """(tau, rho, floor) of the header for an n-point plan"""
    lg = math.log2(n) if n > 1 else 0.0
    p = path_of(n)
    if p == FRAMES:
        t = 4 * lg * U64
        return t, t, 16 * n * TINY
    if p == TWOSTEP:
        t = (4 * lg + 4) * U64
        return t, t, 16 * n * TINY
    if p == DIRECT:
        t = (3 * n + 1) * U64
        return t, math.sqrt(n) * t, 16 * n * TINY
    m = chirp_m(n)
    t = math.sqrt(2 * n - 1) * (8 * math.log2(m) + 12) * U64 + 8 * U64
    return t, math.sqrt(2) * t, 64 * m * math.sqrt(2 * n) * TINY


def exact(x, n, inverse):
    """the transform of each n-point frame of x (complex128), as clongdouble"""
    import scipy.fft

    f = np.asarray(x, np.complex128).reshape(-1, n).astype(np.clongdouble)
    if inverse:
        return scipy.fft.ifft(f, axis=1, norm="forward")
    return scipy.fft.fft(f, axis=1)


def check(got, x, n, inverse, what="", ratios=None):
    """Every bin of every frame of `got` against the header's bound; frames with a non-finite input must be entirely
    non-finite, all others finite.  Returns the worst (per-bin, per-frame) error / bound ratios."""
    tau, rho, floor = constants(n)
    g = np.asarray(got, np.complex128).reshape(-1, n)
    xs = np.asarray(x, np.complex128).reshape(-1, n)
    bad = ~np.isfinite(xs).all(axis=1)
    if bad.any():
        assert not np.isfinite(g[bad]).all(axis=1).any() and (~np.isfinite(g[bad])).all(), (what, "non-finite frame")
    good = ~bad
    assert np.isfinite(g[good]).all(), (what, "finite frame gave a non-finite bin")
    worst_bin = worst_frame = 0.0
    if good.any():
        ref = exact(xs[good], n, inverse)
        s = np.abs(xs[good].astype(np.clongdouble)).sum(axis=1)
        err = np.abs(g[good].astype(np.clongdouble) - ref)
        lim = np.broadcast_to((tau + REF_TAU) * s[:, None] + floor, err.shape)
        r = (err / lim).astype(np.float64)
        worst_bin = float(r.max())
        i = np.unravel_index(int(np.argmax(r)), r.shape)
        assert worst_bin <= 1.0, (what, "bin", i, float(err[i]), float(lim[i]))
        fe = np.sqrt((err ** 2).sum(axis=1))  # long double: frames scaled by 2^500 do not overflow
        fx = np.sqrt((np.abs(ref) ** 2).sum(axis=1))
        flim = (rho + REF_TAU) * fx + math.sqrt(n) * floor
        rf = (fe / flim).astype(np.float64)
        worst_frame = float(rf.max())
        assert worst_frame <= 1.0, (what, "frame", int(np.argmax(rf)))
    if ratios is not None:
        key = (path_of(n), n)
        b, f = ratios.get(key, (0.0, 0.0))
        ratios[key] = (max(b, worst_bin), max(f, worst_frame))
    return worst_bin, worst_frame


def emul_lib(build_dir):
    """Compile tests/emul/fft_f64_emul.cpp into build_dir and return the ctypes handle."""
    import ctypes as C
    import subprocess

    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "fft_f64_emul.cpp")
    so = os.path.join(str(build_dir), "libfft64emul.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", src, "-o", so],
                   check=True)
    lib = C.CDLL(so)
    lib.fft64_emul.restype = C.c_int
    lib.fft64_emul.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    return lib


def emulate(lib, x, n, inverse=False, mutation=0):
    """the plan's output bits for the frames of x (complex128)"""
    xs = np.ascontiguousarray(np.asarray(x, np.complex128).reshape(-1))
    assert len(xs) % n == 0
    y = np.empty_like(xs)
    p = lib.fft64_emul(xs.ctypes.data, n, len(xs) // n, int(bool(inverse)), int(mutation), y.ctypes.data)
    assert p == path_of(n), (n, p)
    return y


def same_bits(a, b):
    a = np.ascontiguousarray(a, np.complex128).view(np.uint64)
    b = np.ascontiguousarray(b, np.complex128).view(np.uint64)
    an = np.isnan(np.ascontiguousarray(a).view(np.float64))
    bn = np.isnan(np.ascontiguousarray(b).view(np.float64))
    return bool(np.array_equal(an, bn) and np.array_equal(a[~an], b[~bn]))
