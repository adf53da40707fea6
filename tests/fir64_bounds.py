"""Per-output error bound of the Complex<f64> FIR (cb_fir_f64, include/comms_b200.h) and the ctypes wrapper of its CPU
emulation (tests/emul/fir_f64_emul.cpp), shared by tests/test_fir_f64_cpu.py and tests/test_gpu_fir_f64.py."""
import os

import numpy as np

U64 = 2.0 ** -53

# ---------------------------------------------------------------- Complex<f64> FIR (cb_fir_f64)
# Every output is two FMA chains over its K_n taps in ascending order (include/comms_b200.h).  With
# A_n = sum |h_k| |x_{n-k}| over those taps:  |y_n - y_exact| <= C_FIR64 K_n u64 A_n + K_n FIR64_FLOOR.  The constant is
# gamma_{2K} on each chain (each term |h.re x.re| + |h.im x.im| <= |h| |x|; sqrt 2 * 2 < 3); the floor covers the
# subnormal range, where an FMA's rounding is absolute (2^-1075 per step, two steps per term).
C_FIR64 = 3.0
FIR64_FLOOR = 2.0 ** -1072


def fir64_bound(kn, amag):
    return C_FIR64 * np.asarray(kn, np.float64) * U64 * np.asarray(amag, np.float64) + np.asarray(kn, np.float64) * FIR64_FLOOR


def fir64_emul_lib(build_dir):
    """Compile tests/emul/fir_f64_emul.cpp into build_dir and return the ctypes handle."""
    import ctypes as C
    import subprocess

    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "fir_f64_emul.cpp")
    so = os.path.join(str(build_dir), "libfir64emul.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", src, "-lquadmath",
                    "-o", so], check=True)
    lib = C.CDLL(so)
    vp, sz = C.c_void_p, C.c_size_t
    lib.fir64_emul.restype = C.c_long
    lib.fir64_emul.argtypes = [vp, sz, vp, sz, C.c_int, C.c_uint, C.c_uint, vp, vp, sz, C.c_int, C.c_int,
                               vp, vp, vp, vp, vp, vp, vp, sz]
    return lib


class Fir64Emul:
    """Result of one emulated stream: y (complex128, the device bits), and with exact=True the exact value
    (exact_hi + exact_lo), err = |y - exact|, amag = A_n; always kn = K_n and bad (the chain reaches a non-finite
    sample)."""

    def __init__(self, lib, taps, x, calls=None, state=None, decim=1, interp=1, mutation=0, exact=True):
        import ctypes as C

        t = np.ascontiguousarray(np.asarray(taps, np.complex128))
        xs = np.ascontiguousarray(np.asarray(x, np.complex128))
        calls = [len(xs)] if calls is None else list(calls)
        assert sum(calls) == len(xs)
        st = None if state is None else np.ascontiguousarray(np.asarray(state, np.complex128))
        D, L = max(int(decim), 1), max(int(interp), 1)
        cap = sum(-(-(m * L) // D) for m in calls) + len(calls) + 1
        cl = np.asarray(calls, np.uint64)
        self.y = np.zeros(cap, np.complex128)
        self.exact_hi = np.zeros(cap, np.complex128) if exact else None
        self.exact_lo = np.zeros(cap, np.complex128) if exact else None
        self.err = np.zeros(cap, np.float64) if exact else None
        self.amag = np.zeros(cap, np.float64) if exact else None
        self.kn = np.zeros(cap, np.uint32)
        self.bad = np.zeros(cap, np.uint8)
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
        n = lib.fir64_emul(p(t), len(t), p(st), 0 if st is None else len(st), int(st is not None), D, L, p(xs), p(cl),
                           len(cl), int(mutation), int(bool(exact)), p(self.y), p(self.exact_hi), p(self.exact_lo),
                           p(self.err), p(self.amag), p(self.kn), p(self.bad), cap)
        if n == -1:
            raise ValueError("off-grid interp state")
        assert n >= 0
        self.n = n
        for k in ("y", "exact_hi", "exact_lo", "err", "amag", "kn", "bad"):
            v = getattr(self, k)
            if v is not None:
                setattr(self, k, v[:n])
        self.bad = self.bad.astype(bool)

    def bound(self):
        return fir64_bound(self.kn, self.amag)

    def ratio(self):
        """worst err / bound over the finite outputs with a non-zero bound (0 if none)"""
        ok = ~self.bad
        b = self.bound()[ok]
        e = self.err[ok]
        nz = b > 0
        return float(np.max(e[nz] / b[nz])) if nz.any() else 0.0


def fir64_check(got, emu, what=""):
    """Every output of `got` equals the emulation bit for bit (NaN positions compared as NaN), is non-finite exactly
    where its chain reaches a non-finite sample, and (when the emulation computed exact values) meets the bound."""
    got = np.asarray(got, np.complex128)
    assert got.shape == emu.y.shape, (what, got.shape, emu.y.shape)
    g = got.view(np.float64).reshape(-1, 2)
    e = emu.y.view(np.float64).reshape(-1, 2)
    nan_g, nan_e = np.isnan(g), np.isnan(e)
    same = (g.view(np.uint64) == e.view(np.uint64)) | (nan_g & nan_e)
    bad = np.flatnonzero(~same.all(axis=1))
    assert bad.size == 0, f"{what}: {bad.size} outputs differ from the emulation, first at {bad[0]}: " \
                          f"got {got[bad[0]]!r}, emulated {emu.y[bad[0]]!r}"
    nonfin = ~np.isfinite(g).all(axis=1)
    wrong = np.flatnonzero(nonfin != emu.bad)
    assert wrong.size == 0, f"{what}: output {wrong[0]} non-finite={nonfin[wrong[0]]}, reaches a non-finite " \
                            f"sample={emu.bad[wrong[0]]}"
    if emu.err is not None:
        fin = ~emu.bad
        over = np.flatnonzero(fin & ~(emu.err <= emu.bound()))
        assert over.size == 0, f"{what}: output {over[0]} error {emu.err[over[0]]:.3e} > bound {emu.bound()[over[0]]:.3e}"
        zero = fin & (emu.amag == 0)
        assert (g[zero] == 0).all(), f"{what}: an output with A_n = 0 is not exactly 0"
