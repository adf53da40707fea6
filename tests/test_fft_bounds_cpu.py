"""The FFT and overlap-save bounds of tests/bounds.py, without a GPU: where their constants come from (the CPU emulation
of the device's FFT passes and of the fused chirp-z kernel; a NumPy f32 emulation of the chirp-z sequence up to
M = 2^20 shows that its error does not grow with N), that the float64 reference is right,
and that they reject single wrong bins, a wrong intermediate, swapped bins, a zero frame that is not zero and a wrong
overlap-save output at a frame seam, all of which the relative-L2 (<= 1e-4 per frame, 2e-5 per FIR call) and
Parseval checks of the parity tests accept."""
import os
import re
import subprocess

import numpy as np
import pytest

import bounds as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a = np.asarray(a).astype(np.complex128).ravel()
    b = np.asarray(b).astype(np.complex128).ravel()
    d = np.linalg.norm(b)
    return np.linalg.norm(a - b) / d if d > 0 else np.linalg.norm(a - b)


def parseval_ok(got, x, n):  # the per-frame energy check of the parity tests
    e_in = (np.abs(np.asarray(x).reshape(-1, n).astype(np.complex128)) ** 2).sum(axis=1)
    e_out = (np.abs(np.asarray(got).reshape(-1, n).astype(np.complex128)) ** 2).sum(axis=1)
    return bool(np.all(np.abs(e_out / (n * e_in) - 1) < 1e-5))


def rnd_c32(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


# ------------------------------------------------------------------ reference
@pytest.mark.parametrize("n", [1, 2, 3, 5, 8, 10, 16, 100, 128, 129, 256])
@pytest.mark.parametrize("inverse", [False, True])
def test_fft64_matches_direct_dft(n, inverse):
    rng = np.random.default_rng(n)
    x = rnd_c32(rng, 3 * n)
    k = np.arange(n)
    W = np.exp((1j if inverse else -1j) * 2 * np.pi * ((k[:, None] * k[None, :]) % n) / n)
    want = x.reshape(3, n).astype(np.complex128) @ W.T
    got = B.fft64(x, n, inverse)
    assert np.abs(got - want).max() <= 1e-13 * np.abs(x).sum(axis=-1).max()


def test_fft_paths_and_constants():
    assert [B.fft_path(n) for n in (1, 2, 3, 4, 7, 8, 100, 127, 128, 129, 4097, 1 << 20)] == \
        ["direct"] * 5 + ["pow2", "direct", "direct", "pow2", "chirpz", "chirpz", "pow2"]
    assert B.fft_path(4095, direct=True) == "direct" and B.fft_path(4097, direct=True) == "chirpz"
    assert [B.chirpz_m(n) for n in (3, 129, 4097, 300000)] == [256, 512, 16384, 1 << 20]
    for l in range(3, 21):  # 50 times tighter than the parity tests' 1e-4 at every size
        assert B.fft_constants(1 << l, "pow2")[1] <= 2e-6


# ------------------------------------------------------------------ calibration: CPU emulation of the device passes
@pytest.fixture(scope="module")
def emul_ratios(tmp_path_factory):
    exe = tmp_path_factory.mktemp("emul") / "fft2_emul"
    src = os.path.join(ROOT, "tests", "emul", "fft2_emul.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I/usr/local/cuda/include", src, "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    rows = [l for l in r.stdout.splitlines() if l.startswith(("fft2 ratio", "chirpz ratio"))]
    return [dict(kind=l.split()[2] if l.startswith("fft2") else "chirpz",
                 **{k: float(v) for k, v in re.findall(r"(\w+)=([0-9.]+)", l)}) for l in rows]


def test_emulated_device_fft_within_constants(emul_ratios):
    # every single-CTA size 16 .. 16384 and the 256 x 256 two-step form of 65536 points (twiddle16c), both directions
    emul_ratios = [r for r in emul_ratios if r["kind"] != "chirpz"]
    sizes = {(int(r["N"]), int(r["inv"])) for r in emul_ratios}
    assert sizes == {(1 << l, i) for l in list(range(4, 15)) + [16] for i in (0, 1)}
    wbin = max(max(r["impulse_bin"], r["tone_bin"], r["random_bin"]) for r in emul_ratios)
    wnorm = max(max(r["impulse_norm"], r["tone_norm"], r["random_norm"]) for r in emul_ratios)
    assert wbin <= B.C_TAU and wnorm <= B.C_RHO, (wbin, wnorm)
    # the constants sit at most 2x above the worst emulated ratio, and that worst case is a real one (not noise)
    assert B.C_TAU <= 2 * wbin and B.C_RHO <= 2 * wnorm and wbin > 1 and wnorm > 0.5, (wbin, wnorm)


# ------------------------------------------------------------------ calibration: chirp-z
def test_emulated_device_chirpz_within_constants(emul_ratios):
    # the fused chirp-z kernel on the device's M-point passes, M = 512 .. 16384, both directions: these ratios set
    # C_CHIRPZ and C_CHIRPZ_RHO
    cz = [r for r in emul_ratios if r["kind"] == "chirpz"]
    assert {(int(r["N"]), int(r["inv"])) for r in cz} == {(n, i) for n in (129, 1000, 4095, 4097, 8191) for i in (0, 1)}
    for r in cz:
        assert int(r["M"]) == B.chirpz_m(int(r["N"])), r
    wbin, wnorm = max(r["bin"] for r in cz), max(r["norm"] for r in cz)
    assert wbin <= B.C_CHIRPZ and wnorm <= B.C_CHIRPZ_RHO, (wbin, wnorm)
    assert B.C_CHIRPZ <= 2 * wbin and B.C_CHIRPZ_RHO <= 2 * wnorm, (wbin, wnorm)


def chirpz_setup(n, inverse):
    """the chirp w (f32) and the f32-rounded spectrum B of the wrapped conj chirp, as bluestein_setup (api.cu) builds
    them: i^2 reduced mod 2N in integers, angles and B in float64"""
    m = B.chirpz_m(n)
    i = np.arange(n, dtype=np.int64)
    a = (1.0 if inverse else -1.0) * np.pi * ((i * i) % (2 * n)) / n
    w64 = np.exp(1j * a)
    b = np.zeros(m, np.complex128)
    b[:n] = np.conj(w64)
    b[m - np.arange(1, n)] = np.conj(w64[1:])
    return w64.astype(np.complex64), np.fft.fft(b).astype(np.complex64), m


def chirpz_emul(x, n, inverse):
    """the chirp-z sequence in f32: a = x w (zero-padded to M), M-point transform, times B, inverse M-point
    transform, times w, times 1/M (NumPy's single-precision transforms stand in for the M-point plans)"""
    w, bs, m = chirpz_setup(n, inverse)
    x = np.asarray(x, np.complex64).reshape(-1, n)
    a = np.zeros((x.shape[0], m), np.complex64)
    a[:, :n] = x * w
    A = np.fft.fft(a, axis=1).astype(np.complex64) * bs
    c = (np.fft.ifft(A, axis=1) * np.float32(m)).astype(np.complex64)  # unnormalised inverse
    return (c[:, :n] * w * np.float32(1.0 / m)).astype(np.complex64).ravel()


def _chirpz_frames(rng, n):
    imp = np.zeros((6, n), np.complex64)
    for j, p in enumerate((0, 1, n // 2, n - 1, n // 3, 7)):
        imp[j, p] = 1
    k = np.arange(n)
    tones = np.stack([np.exp(2j * np.pi * (k0 * k % n) / n) for k0 in (1, n // 5 + 2)]).astype(np.complex64)
    return np.concatenate([imp, tones, rnd_c32(rng, 4 * n).reshape(4, n)])


@pytest.mark.parametrize("n", [129, 1000, 4095, 4097, 10007, 65535, 300000])
@pytest.mark.parametrize("inverse", [False, True])
def test_emulated_chirpz_within_constants(n, inverse):
    rng = np.random.default_rng(n + inverse)
    x = _chirpz_frames(rng, n)
    got = chirpz_emul(x, n, inverse)
    fails, wbin, wnorm = B.fft_bound_report(got, x, n, inverse, "chirpz")
    assert not fails, fails[:3]
    # NumPy's f32 transforms are more accurate than the device's passes: in units of u log2(M) S_f and u log2(M) ||X||
    # this reaches 0.72 and 0.29, flat from N = 129 to 300000 (M = 2^20), against 2.74 and 1.00 for the device passes
    assert wbin * B.C_CHIRPZ <= 0.8 and wnorm * B.C_CHIRPZ_RHO <= 0.32, (wbin * B.C_CHIRPZ, wnorm * B.C_CHIRPZ_RHO)


# ------------------------------------------------------------------ the bounds accept what is right ...
@pytest.mark.parametrize("n", [8, 256, 4096, 65536])
def test_f32_rounded_exact_passes(n):
    rng = np.random.default_rng(n)
    x = rnd_c32(rng, 4 * n)
    x[n:2 * n] = 0
    x[2 * n:3 * n] *= np.float32(2.0 ** -140)  # subnormal frame: the absolute floor
    for inverse in (False, True):
        X = B.fft64(x, n, inverse)
        assert not B.fft_bound_report(X.astype(np.complex64), x, n, inverse)[0]


def test_nonfinite_frames_are_isolated():
    n = 256
    rng = np.random.default_rng(9)
    x = rnd_c32(rng, 4 * n)
    x[n + 5] = np.inf
    x[2 * n + 7] = np.nan
    X = B.fft64(x, n).astype(np.complex64).ravel()
    assert not B.fft_bound_report(X, x, n)[0]
    bad = X.copy()
    bad[n + 9] = 1  # a finite bin in the Inf frame
    assert "holds a non-finite input" in B.fft_bound_report(bad, x, n)[0][0]
    bad = X.copy()
    bad[3 * n + 1] = np.nan  # a neighbour of the NaN frame
    assert "frame 3 (finite input)" in B.fft_bound_report(bad, x, n)[0][0]


# ------------------------------------------------------------------ ... and reject what the old checks let through
def test_mutation_one_bin_off_by_1e3():
    n = 65536
    rng = np.random.default_rng(1)
    x = rnd_c32(rng, n)
    X = B.fft64(x, n)[0]
    got = X.astype(np.complex64)
    k = 12345
    got[k] = X[k] * (1 + 1e-3)
    assert rel_l2(got, X) <= 1e-4 and parseval_ok(got, x, n)
    fails = B.fft_bound_report(got, x, n)[0]
    assert fails and "frame 0" in fails[0]


def test_mutation_one_intermediate_of_a_256x256_split():
    # X[k1 + 256 k2] = sum_n2 W_256^{n2 k2} (W_N^{n2 k1} Y[k1][n2]),  Y[k1][n2] = sum_n1 x[256 n1 + n2] W_256^{n1 k1}
    n, d = 65536, 1e-3
    rng = np.random.default_rng(2)
    x = rnd_c32(rng, n).astype(np.complex128)
    Y = np.fft.fft(x.reshape(256, 256), axis=0)  # Y[k1, n2]
    Y[77, 200] *= 1 + d
    k1, n2 = np.arange(256)[:, None], np.arange(256)[None, :]
    Z = Y * np.exp(-2j * np.pi * k1 * n2 / n)
    got = np.fft.fft(Z, axis=1).T.ravel().astype(np.complex64)  # [k2, k1] -> k1 + 256 k2
    X = B.fft64(x, n)[0]
    assert rel_l2(got, X) <= 1e-4 and parseval_ok(got, x, n)
    Y[77, 200] /= 1 + d  # the unperturbed split passes
    good = np.fft.fft(Y * np.exp(-2j * np.pi * k1 * n2 / n), axis=1).T.ravel().astype(np.complex64)
    assert not B.fft_bound_report(good, x, n)[0]
    fails = B.fft_bound_report(got, x, n)[0]
    assert fails and "||err||/(rho ||X||)" in fails[-1]


def test_mutation_two_bins_swapped():
    n = 4096
    rng = np.random.default_rng(3)
    x = rnd_c32(rng, 8 * n)
    got = B.fft64(x, n).astype(np.complex64).ravel()
    got[5 * n + 10], got[5 * n + 11] = got[5 * n + 11], got[5 * n + 10]
    assert parseval_ok(got, x, n)  # an unsampled frame: only its energy was checked
    fails = B.fft_bound_report(got, x, n)[0]
    assert fails and fails[0].startswith("pow2 N=4096 forward: frame 5 bin 1") and "(2 of 4096 bins outside)" in fails[0]


def test_mutation_zero_frame_not_zero():
    n = 1024
    x = np.zeros(3 * n, np.complex64)
    x[:n] = 1
    got = B.fft64(x, n).astype(np.complex64).ravel()
    got[n:2 * n] = 1e-30
    assert rel_l2(got[n:2 * n], np.zeros(n)) <= 1e-4
    fails = B.fft_bound_report(got, x, n)[0]
    assert fails and "frame 1 is all zeros" in fails[0]


def test_mutation_overlap_save_seam_output():
    # a loud random call; the frame starting at output f * hop holds only the K samples its first output sees, matched
    # to the taps, so that this output is as large as ||H||_inf ||x_f|| allows
    K, f = 129, 3
    hop = B.OLS_N - (K - 1)
    rng = np.random.default_rng(4)
    k = np.arange(K)
    taps = (np.exp(1j * np.pi * k * k / K) / np.sqrt(K)).astype(np.complex64)  # chirp: |H| nearly flat
    n = 8 * hop
    x = rnd_c32(rng, n)
    s0 = f * hop - (K - 1)
    x[s0:s0 + B.OLS_N] = 0
    x[s0:s0 + K] = np.conj(taps[::-1])
    want, _ = B.fir64(x, taps)
    got = want.astype(np.complex64)
    bound, fr = B.ols_bound(x, taps)
    assert np.all(np.abs(got - want) <= bound) and fr[f * hop] == f
    seam = f * hop
    assert seam in B.ols_seams(n, K)
    got[seam] = want[seam] * (1 + 1e-4)
    assert rel_l2(got, want) <= 2e-5  # the per-call check of the parity tests
    assert np.abs(got[seam] - want[seam]) > bound[seam]
