"""The Complex<f64> FIR's numerical contract (include/comms_b200.h, cb_fir_f64) without a GPU: the CPU emulation of its
operation order (tests/emul/fir_f64_emul.cpp) and its __float128 reference against Fraction, the bound
|y_n - y_exact| <= 3 K_n u A_n + K_n 2^-1072 on random and adversarial inputs (and for the oracle's plain complex128
arithmetic), and defects that the bound and the bit-exact comparison reject while a relative-L2 check accepts them.
"""
import os
import re
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import fir64_bounds as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53
L2_TOL = 1e-5  # the relative-L2 tolerance the f32 parity checks use


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return B.fir64_emul_lib(tmp_path_factory.mktemp("fir64_emul"))


def rnd(rng, n, scale=1.0):
    return scale * (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n))


def rel_l2(got, want):
    """relative L2 over the outputs finite in both (what a check that tolerates non-finite inputs compares)"""
    n = min(len(got), len(want))
    g, w = got[:n], want[:n]
    ok = np.isfinite(g) & np.isfinite(w)
    return float(np.linalg.norm(g[ok] - w[ok]) / np.linalg.norm(w[ok]))


def rejects(got, emu):
    try:
        B.fir64_check(got, emu, "mutant")
    except AssertionError:
        return True
    return False


# --------------------------------------------------------------------------------------------- the exact reference
def _fraction_conv(t, x, state, n):
    s = list(state[::-1]) + list(x)  # chronological
    H = len(state)
    out = []
    for i in range(n):
        re = im = Fraction(0)
        for k in range(min(len(t), len(state))):
            h, v = t[k], s[H + i - k]
            hr, hi, vr, vi = (Fraction(float(z)) for z in (h.real, h.imag, v.real, v.imag))
            re += hr * vr - hi * vi
            im += hr * vi + hi * vr
        out.append((re, im))
    return out


@pytest.mark.parametrize("case", ["random", "dyadic", "wide"])
def test_float128_reference_matches_fraction(emul, case):
    rng = np.random.default_rng({"random": 1, "dyadic": 2, "wide": 3}[case])
    k, n = 9, 40
    if case == "dyadic":
        t = (rng.integers(-64, 64, k) + 1j * rng.integers(-64, 64, k)) / 32.0
        x = (rng.integers(-1024, 1024, n) + 1j * rng.integers(-1024, 1024, n)) / 256.0
    elif case == "wide":
        t = rnd(rng, k) * 2.0 ** rng.integers(-40, 40, k)
        x = rnd(rng, n) * 2.0 ** rng.integers(-60, 60, n)
    else:
        t, x = rnd(rng, k), rnd(rng, n)
    st = rnd(rng, k)
    emu = B.Fir64Emul(emul, t, x, state=st)
    want = _fraction_conv(t, x, st, n)
    for i, (re, im) in enumerate(want):
        for got_hi, got_lo, w in ((emu.exact_hi[i].real, emu.exact_lo[i].real, re),
                                  (emu.exact_hi[i].imag, emu.exact_lo[i].imag, im)):
            d = abs(Fraction(float(got_hi)) + Fraction(float(got_lo)) - w)
            if case == "dyadic":
                assert d == 0, (i, float(d))
            else:  # quad rounding of the sum: far below one f64 ulp of A_n
                assert d <= Fraction(float(emu.amag[i])) * Fraction(1, 1 << 100), (i, float(d))


# ------------------------------------------------------------------------------------------------------ the bound
@pytest.mark.parametrize("k,real,D,L", [(64, True, 1, 1), (64, False, 1, 1), (1025, False, 1, 1), (63, True, 5, 1),
                                        (1024, True, 1, 8), (47, False, 2, 3)])
def test_emulation_meets_the_bound_on_random_inputs(emul, k, real, D, L):
    rng = np.random.default_rng(k + D + L)
    t = rnd(rng, k).real.astype(np.complex128) if real else rnd(rng, k)
    x = rnd(rng, 20000 if k < 1000 else 3000)
    emu = B.Fir64Emul(emul, t, x, calls=[len(x) // 3, len(x) - len(x) // 3], decim=D, interp=L)
    r = emu.ratio()
    print(f"fir_f64 emulated worst bound ratio, random, K={k} {'real' if real else 'complex'} D={D} L={L}: {r:.3e}")
    assert 0 < r <= 1.0


def _adversarial(K):
    # one output whose every FMA rounds the same way: real taps of 1, and terms 1 + 0.49 ulp(running sum), so that each
    # addition drops just under half an ulp
    x = np.zeros(K, np.complex128)
    acc = 0.0
    for k in range(K):
        v = 1.0 + 0.49 * np.spacing(acc + 1.0)
        x[K - 1 - k] = complex(v, v)
        acc += v
    return np.ones(K, np.complex128), x


@pytest.mark.parametrize("K", [64, 1025, 4097])
def test_emulation_meets_the_bound_on_adversarial_inputs(emul, K):
    t, x = _adversarial(K)
    emu = B.Fir64Emul(emul, t, x)
    r = float(emu.err[K - 1] / emu.bound()[K - 1])
    print(f"fir_f64 emulated bound ratio, one-way roundings, K={K}: {r:.3f}")
    assert 0.1 < r <= 1.0  # the roundings do accumulate, and stay within the bound


def test_oracle_complex128_meets_the_bound(emul):
    import oracle

    oracle.build()
    rng = np.random.default_rng(4)
    for k in (1, 64, 1025):
        t, x, st = rnd(rng, k), rnd(rng, 5000), rnd(rng, k)
        got, _ = oracle.batch_fir(x, t, st)
        emu = B.Fir64Emul(emul, t, x, state=st)
        ex = emu.exact_hi + emu.exact_lo
        err = np.abs(got - ex)
        r = float(np.max(err / emu.bound()))
        print(f"oracle.batch_fir complex128 (no FMA) worst bound ratio, K={k}: {r:.3e}")
        assert r <= 1.0


# ----------------------------------------------------------------------------------------------------- mutations
def test_one_output_off_by_2_20_ulp_is_rejected(emul):
    rng = np.random.default_rng(5)
    t, x = rnd(rng, 64), rnd(rng, 1 << 16)
    emu = B.Fir64Emul(emul, t, x)
    got = emu.y.copy()
    i = 40000
    got[i] = complex(got[i].real + np.spacing(got[i].real) * 2.0 ** 20, got[i].imag)
    assert rel_l2(got, emu.y) < L2_TOL
    assert rejects(got, emu)
    B.fir64_check(emu.y, emu, "unmutated")


def test_missing_halo_term_at_a_tile_seam_is_rejected(emul):
    rng = np.random.default_rng(6)
    t = rnd(rng, 64)
    t[1] *= 1e-4  # a quiet tap, so that a relative-L2 check cannot see the missing term
    x = rnd(rng, 1 << 16)
    emu = B.Fir64Emul(emul, t, x)
    mut = B.Fir64Emul(emul, t, x, mutation=1).y
    assert rel_l2(mut, emu.y) < L2_TOL
    assert rejects(mut, emu)


def test_dropped_last_tap_is_rejected(emul):
    rng = np.random.default_rng(7)
    t = rnd(rng, 64)
    t[63] *= 1e-6
    x = rnd(rng, 1 << 14)
    emu = B.Fir64Emul(emul, t, x)
    mut = B.Fir64Emul(emul, t, x, mutation=2).y
    assert rel_l2(mut, emu.y) < L2_TOL
    assert rejects(mut, emu)


def test_second_call_from_a_zero_history_is_rejected(emul):
    rng = np.random.default_rng(8)
    t = rnd(rng, 64)
    x = rnd(rng, 1 << 15)
    x[(1 << 14) - 64: 1 << 14] *= 1e-4  # the first call ends quietly
    calls = [1 << 14, 1 << 14]
    emu = B.Fir64Emul(emul, t, x, calls=calls)
    mut = B.Fir64Emul(emul, t, x, calls=calls, mutation=3).y
    assert rel_l2(mut, emu.y) < L2_TOL
    assert rejects(mut, emu)


def test_padding_tap_times_inf_is_rejected(emul):
    rng = np.random.default_rng(9)
    t = rnd(rng, 63)  # padded to 64 by the mutant
    x = rnd(rng, 1 << 14)
    x[5000] = np.inf
    emu = B.Fir64Emul(emul, t, x)
    mut = B.Fir64Emul(emul, t, x, mutation=4).y
    assert np.isnan(mut[5000 + 63]) and np.isfinite(emu.y[5000 + 63])
    assert rel_l2(mut, emu.y) < L2_TOL
    assert rejects(mut, emu)


def test_decimation_phase_carried_over_calls_is_rejected(emul):
    n = 2001
    f = 1e-7  # a slow tone: neighbouring outputs differ by ~2 pi f of themselves
    x = np.exp(2j * np.pi * f * np.arange(n))
    t = np.full(8, 0.125, np.complex128)
    calls = [1001, 1000]
    emu = B.Fir64Emul(emul, t, x, calls=calls, decim=2)
    mut = B.Fir64Emul(emul, t, x, calls=calls, decim=2, mutation=5).y
    assert len(mut) == len(emu.y)
    assert rel_l2(mut, emu.y) < L2_TOL
    assert rejects(mut, emu)


# ------------------------------------------------------------------------------------------------ header, build
def test_header_states_the_constants_the_tests_enforce():
    h = open(os.path.join(ROOT, "include", "comms_b200.h")).read()
    assert "|y_n - y_exact| <= 3 K_n u A_n + K_n 2^-1072" in h
    assert "u = 2^-53" in h
    assert B.C_FIR64 == 3.0 and B.FIR64_FLOOR == 2.0 ** -1072
    for fn in ("re = fma(h.re, x.re, re); re = fma(-h.im, x.im, re); im = fma(h.re, x.im, im); im = fma(h.im, x.re, im)",
               "re = fma(h.re, x.re, re); im = fma(h.re, x.im, im)"):
        assert fn in h


def test_new_kernels_have_no_stack_frame():
    lib = os.path.join(ROOT, "comms-rs_b200", "libcomms_b200.so")
    if not os.path.exists(lib):
        pytest.skip("library not built")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.dirname(nvcc))
    if cuobjdump is None:
        pytest.skip("cuobjdump not found on PATH or beside nvcc")
    out = subprocess.run([cuobjdump, "--dump-resource-usage", lib], capture_output=True, text=True, check=True).stdout
    usage = {m.group(1): (int(m.group(2)), int(m.group(3)))
             for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out)}
    hits = {k: v for k, v in usage.items() if "fir64_stream_kernel" in k or "fir64_resample_kernel" in k}
    assert len(hits) == 4, sorted(hits)
    for name, (regs, stack) in hits.items():
        assert stack == 0, (name, stack)
        if "stream" in name:  # 256 threads x 2 CTAs per SM (__launch_bounds__(256, 2))
            assert regs * 256 * 2 <= 65536, (name, regs)


def test_cpp_nodes_compile(tmp_path):
    src = tmp_path / "f64_nodes.cpp"
    src.write_text('#include "comms_b200_nodes.hpp"\n'
                   "using namespace comms_b200;\n"
                   "void use() {\n"
                   "    std::vector<c64> taps(8, c64{1.0, 0.0}), st(8, c64{0.0, 0.0});\n"
                   "    BatchFirNodeF64 a(taps, &st, 2, 1);\n"
                   "    auto r = a.run(taps);\n"
                   "    (void)r;\n"
                   "    PulseNodeF64 p(taps, 4);\n"
                   "    auto q = p.run(taps[0]);\n"
                   "    (void)q;\n"
                   "    (void)a.state();\n"
                   "}\n")
    subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(ROOT, "comms-rs_b200", "host"), str(src)], check=True)
