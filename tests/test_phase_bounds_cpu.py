"""The phase-law and f64-estimator bounds of tests/bounds.py, without a GPU: the exact-phase reference against mpmath,
the constants against the CPU emulation of the device's f64 operation order (tests/emul/phase_emul.cpp), the NCO's
causal prefix order (the order it used before fails the causal bound on one huge or non-finite phase error), and
mutations that the new bounds reject while the earlier checks accept them.

The mixer's f32 part is not emulated: it rests on sincosf's documented 2 ulp (see C_MIX in tests/bounds.py)."""
import json
import os
import subprocess
from fractions import Fraction

import mpmath
import numpy as np
import pytest

import bounds as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------- the exact-phase reference
def _mp_phase(phase0, dphase, k, prefix=0.0):
    mpmath.mp.prec = 300
    t = mpmath.mpf(phase0) + mpmath.mpf(int(k)) * mpmath.mpf(dphase) + mpmath.mpf(prefix)
    tp = 2 * mpmath.pi
    return t - tp * mpmath.nint(t / tp)


@pytest.mark.parametrize("dphase", [0.37, 2.0 ** -40, 2 * np.pi - 2.0 ** -40, np.nextafter(2 * np.pi, 0), np.pi])
@pytest.mark.parametrize("phase0", [0.0, -3.0, 1e6])
def test_phase_exact_matches_mpmath(dphase, phase0):
    rng = np.random.default_rng(1)
    k = np.concatenate([[0, 1, 2, 2047, 2048, (1 << 21) + 5, (1 << 28) - 1, (1 << 29) - 1, (1 << 29) - 2],
                        rng.integers(0, 1 << 29, 40)]).astype(np.int64)
    pre = np.where(np.arange(len(k)) % 2, rng.integers(-(1 << 52), 1 << 52, len(k)) * 2.0 ** -40, 0.0)
    h, l = B.phase_exact(phase0, dphase, k, pre)
    mpmath.mp.prec = 300
    for i in range(len(k)):
        want = _mp_phase(phase0, dphase, k[i], float(pre[i]))
        d = mpmath.mpf(float(h[i])) + mpmath.mpf(float(l[i])) - want
        d -= 2 * mpmath.pi * mpmath.nint(d / (2 * mpmath.pi))  # near +-pi either representative is right
        assert abs(d) < mpmath.mpf(2) ** -64, (k[i], float(d))
        assert abs(float(h[i])) <= np.pi + 1e-6  # q = rint(hi / 2 pi) may pick the turn next to the nearest


def test_cis_and_mix_exact_match_mpmath():
    rng = np.random.default_rng(2)
    x = (rng.standard_normal(64) + 1j * rng.standard_normal(64)).astype(np.complex64)
    d, p0, start = 2 * np.pi - 2.0 ** -20, 1e6, (1 << 28) - 64
    er, ei = B.mix_exact(x, d, p0, start)
    mpmath.mp.prec = 300
    for i in range(0, 64, 7):
        t = _mp_phase(p0, d, start + i)
        z = mpmath.mpc(float(x[i].real), float(x[i].imag)) * mpmath.expjpi(t / mpmath.pi)
        assert abs(complex(z) - complex(float(er[i]), float(ei[i]))) < 1e-17 * (1 + abs(x[i]))


def test_exact_prefix_matches_fraction():
    rng = np.random.default_rng(3)
    p = rng.integers(-(1 << 29), 1 << 29, 5000) * 2.0 ** -40
    p[[7, 100, 2047, 4000]] = [1e6, 5e-324, -3.3e-310, 1.0 / 3.0]
    h, l = B.exact_prefix(p)
    acc = Fraction(0)
    for k in range(len(p)):
        acc += Fraction(float(p[k]))
        assert abs(Fraction(float(h[k])) + Fraction(float(l[k])) - acc) <= abs(acc) * Fraction(1, 1 << 100) + \
            Fraction(1, 1 << 1074), k
    q = p.copy()
    q[300] = np.nan
    h, _ = B.exact_prefix(q)
    assert np.isfinite(h[:300]).all() and np.isnan(h[300:]).all()


def test_freq_exact_matches_fraction():
    rng = np.random.default_rng(4)
    x = rng.standard_normal(301) * 2.0 ** rng.integers(-30, 30, 301) + 1j * rng.standard_normal(301)
    S, T, (re, im) = B.freq_exact(x)
    sr = sum(Fraction(float(x[i + 1].real)) * Fraction(float(x[i].real)) +
             Fraction(float(x[i + 1].imag)) * Fraction(float(x[i].imag)) for i in range(300))
    si = sum(Fraction(float(x[i + 1].imag)) * Fraction(float(x[i].real)) -
             Fraction(float(x[i + 1].real)) * Fraction(float(x[i].imag)) for i in range(300))
    scale = Fraction(T)
    assert abs(Fraction(re[0]) + Fraction(re[1]) - sr) <= scale * Fraction(1, 1 << 100)
    assert abs(Fraction(im[0]) + Fraction(im[1]) - si) <= scale * Fraction(1, 1 << 100)


def test_timing_exact_matches_direct_f64_within_its_error():
    # long double reference against a plain f64 evaluation of the reference's formula (f64 error ~ 1e-13 here)
    rng = np.random.default_rng(5)
    N, D, n = 3, 2, 700
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    taps = B.timing_taps(N, D, 0.5)
    S, W = B.timing_exact(x, taps, N, D)
    r = np.cos((-np.pi * np.arange(n)) / N) + 1j * np.sin((-np.pi * np.arange(n)) / N)
    qin, din = np.conj(x) * r, x * r
    qout = np.convolve(qin, taps)[:n]
    dout = np.concatenate([np.zeros(N * D), din[: n - N * D]])
    want = np.cumsum(qout * dout)
    assert np.abs(S.astype(np.complex128) - want).max() <= 1e-12 * W[-1]


# -------------------------------------------------------------------------------------------------- CPU emulation
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    exe = tmp_path_factory.mktemp("phase_emul") / "phase_emul"
    src = os.path.join(ROOT, "tests", "emul", "phase_emul.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", src, "-lquadmath", "-o", str(exe)], check=True)

    def run(*args):
        r = subprocess.run([str(exe)] + [str(a) for a in args], capture_output=True, text=True, check=True)
        return json.loads(r.stdout)

    return run


NCO_CASES = ("phase0", "random", "chain", "random3")


def test_emulated_nco_within_constants(emul):
    res = {c: emul("nco", "fixed", c, B.C_NCO_A, B.C_NCO_B) for c in NCO_CASES}
    for c, r in res.items():
        assert r["outside"] == 0 and r["worst"] <= 1.0, r
    # each constant is at most about twice the worst ratio of the case that exercises its term
    assert res["phase0"]["worst"] >= 0.45, res["phase0"]
    assert res["chain"]["worst"] >= 0.45, res["chain"]


@pytest.mark.parametrize("case", ["huge", "nan"])
def test_emulated_nco_prefix_order_is_causal(emul, case):
    """One perr of 1e6, or one NaN, in the middle of a thread's 8, a warp and a tile: with exclusive prefixes formed
    as incl - v the outputs before it leave the causal bound (NaN, or cancellation at ulp(1e6)); with the shifted
    scan the library now uses they meet it, and every output from the NaN on is NaN."""
    old = emul("nco", "old", case, B.C_NCO_A, B.C_NCO_B)
    new = emul("nco", "fixed", case, B.C_NCO_A, B.C_NCO_B)
    assert old["outside"] > 100 and old["worst"] > 100, old
    assert new["outside"] == 0 and new["worst"] <= 1.0 and new["not_nan_after"] == 0, new


def test_emulated_freq_within_constant(emul):
    res = [emul("freq", c, B.C_FREQ) for c in ("random", "chain", "n3", "n2049")]
    assert all(r["worst"] <= 1.0 for r in res), res
    assert max(r["worst"] for r in res) >= 0.4, res
    assert res[1]["depth"] == B.freq_depth(res[1]["n"]), res[1]


@pytest.mark.parametrize("N,D,n,case", [(10, 5, 20000, "qpsk"), (10, 5, 20000, "noise"), (3, 2, 5000, "noise"),
                                        (8, 0, 3000, "noise"), (8, 256, 6000, "noise"), (10, 5, 1212417, "noise")])
def test_emulated_timing_within_constant(emul, N, D, n, case):
    r = emul("timing", N, D, n, case, B.C_TIM)
    assert r["worst"] <= 1.0, r


# ------------------------------------------------------------------------------ mutations the bounds must reject
def _nco_ref(n, seed=6, phase0=0.5, dphase=2 * np.pi - 2.0 ** -20):
    rng = np.random.default_rng(seed)
    perr = rng.integers(-(1 << 30) + 1, 1 << 30, n) * 2.0 ** -40
    c, s = B.nco_exact(phase0, dphase, perr)
    S = np.cumsum(np.abs(perr))
    chunks = np.arange(n) // B.NCO_CHUNK
    return perr, c, s, B.nco_bound(phase0, S, 0, chunks)


def _old_nco_check(got, want, n):
    return np.abs(got - want).max() <= 1e-12 + 2e-16 * n * 8  # test_nco_batch_matches_reference_recurrence


def test_nco_bound_rejects_one_output_in_the_second_scan_chunk():
    n = (1 << 21) + 64
    _, c, s, bound = _nco_ref(n)
    exact = (c + 1j * s).astype(np.complex128)
    k = (1 << 21) + 5
    got = exact.copy()
    got[k] *= np.exp(1e-11j)
    assert _old_nco_check(got, exact, n)
    fails, w, r = B.nco_bound_report(got, c, s, bound)
    assert fails and w == k and r > 2, (fails, w, r)
    assert not B.nco_bound_report(exact, c, s, bound)[0]


def test_nco_bound_rejects_a_wrong_chunk_carry():
    n = (1 << 21) + 4096
    _, c, s, bound = _nco_ref(n)
    exact = (c + 1j * s).astype(np.complex128)
    got = exact.copy()
    got[1 << 21:] *= np.exp(1e-11j)
    assert _old_nco_check(got, exact, n)
    fails, w, r = B.nco_bound_report(got, c, s, bound)
    assert fails and w >= 1 << 21 and "4096 of" in fails[0], fails


def test_mixer_bound_rejects_one_output_that_rel_l2_accepts():
    rng = np.random.default_rng(7)
    n = 200001
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    er, ei = B.mix_exact(x, 0.37, 0.5)
    exact = (er + 1j * ei).astype(np.complex128)
    got = exact.astype(np.complex64).astype(np.complex128)
    got[123457] += 1e-4 * abs(x[123457])
    rel = np.linalg.norm(got - exact) / np.linalg.norm(exact)
    assert rel <= 1e-5  # the check of test_gpu_parity
    fails, w, r = B.mix_bound_report(got, x, 0.37, 0.5)
    assert fails and w == 123457 and r > 50, (fails, r)
    assert not B.mix_bound_report(exact.astype(np.complex64), x, 0.37, 0.5)[0]


@pytest.fixture(scope="module")
def freq_big():
    n = (1 << 24) + 5
    rng = np.random.default_rng(8)
    x = np.exp(2j * np.pi * rng.random(n)) * rng.uniform(0.5, 1.5, n)
    return x, B.freq_exact(x)


@pytest.mark.parametrize("drop", ["last", "seam"])
def test_freq_bound_rejects_a_dropped_term(freq_big, drop):
    x, (S, T, (re, im)) = freq_big
    n = len(x)
    i = n - 2 if drop == "last" else 303104 * 7 - 1  # a stride seam at the 1184-block launch
    t = x[i + 1] * np.conj(x[i])
    E = B.C_FREQ * B.U64 * B.freq_depth(n) * T
    ok, ratio, skipped = B.est_bound_report(float(np.angle(S - t)), abs(S), E, B.angle_dd(re, im))
    assert not ok and not skipped and ratio > 100, ratio
    assert B.est_bound_report(float(np.angle(S)), abs(S), E, B.angle_dd(re, im))[0]
    # the earlier long-input check is a pure tone, on which every term is equal: dropping one moves nothing
    tone = np.exp(0.3j * np.arange(4096))
    St = np.sum(tone[1:] * np.conj(tone[:-1]))
    assert abs(np.angle(St - tone[i % 4000 + 1] * np.conj(tone[i % 4000])) - np.angle(St)) < 1e-9


def test_timing_bound_rejects_a_missing_halo_tap_at_a_tile_seam():
    # n > 1184 * 1024: block 0 loops to tile 1184, whose first output needs the oldest tap from the rebuilt halo
    N, D, n = 10, 5, 1212417
    rng = np.random.default_rng(9)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)) / np.sqrt(2)
    taps = B.timing_taps(N, D, 0.5)
    S, W = B.timing_exact(x, taps, N, D)
    i = 1184 * 1024
    m = np.arange(n, dtype=np.float64)
    r = np.cos((-np.pi * m) / N) + 1j * np.sin((-np.pi * m) / N)
    k = len(taps) - 2  # the oldest tap of this filter is -2e-18 (cos(-5 pi / 2) in f64); the next is -1.1e-3
    assert abs(taps[k]) > 1e-3
    dq = taps[k] * np.conj(x[i - k]) * r[i - k] * x[i - N * D] * r[i - N * D]
    exact = complex(S[-1])
    E = B.timing_E(n, len(taps), W[-1])
    scale = -N / (2 * np.pi)
    ok, ratio, _ = B.est_bound_report(scale * np.angle(exact - dq), abs(exact), E, np.angle(exact), scale)
    assert not ok and ratio > 10, ratio
    assert B.est_bound_report(scale * np.angle(exact), abs(exact), E, np.angle(exact), scale)[0]


def test_header_states_the_enforced_constants():
    with open(os.path.join(ROOT, "include", "comms_b200.h")) as f:
        h = " ".join(f.read().split())
    assert B.C_MIX == 13 and "(13 u32 + u64 (|phase| + n dphase + 8 pi + c)) |x[n]| + 2^-148" in h
    assert B.MIX_FLOOR == 2.0 ** -148 and B.mix_carry(1.0, 8, 0.5) == 2 * np.pi + 2.0 ** -9 * 5.0
    assert (B.C_NCO_A, B.C_NCO_B, B.C_SINCOS) == (2.0, 16.0, 6.0)
    assert "u64 (2 (|phase_0| + 2 pi (1 + calls_k + chunks_k)) + 16 S_k + 6)" in h and B.NCO_CHUNK == 1 << 21
    assert B.EST_ABS == 2.0 ** -49 and B.C_FREQ == B.C_TIM == np.sqrt(2.0)
    assert "asin(E / |S|) + 2^-49" in h and "D = m + ceil(P / 256) + 26" in h
    assert B.freq_depth(1 << 24) == -(-((1 << 24) - 1) // (256 * 1184)) + 5 + 26
    assert "E = u64 (sqrt(2) (ntaps4 + D) + 16)" in h and "D = 4 ceil(T / P) + ceil(P / 256) + 26" in h
    assert B.timing_depth(3000, 101) == 4 * 1 + 1 + 26 and 2 * (B.C_SINCOS + 2) == 16
