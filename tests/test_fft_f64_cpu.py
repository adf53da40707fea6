"""The Complex<f64> FFT's numerical contract (include/comms_b200.h, cb_fft_f64) without a GPU: the exact reference
(scipy.fft over clongdouble) against mpmath, the CPU emulation of every path (tests/emul/fft_f64_emul.cpp) against
the header's per-bin and per-frame bounds, the edges, and six planted defects that the check rejects.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import fft64_bounds as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RATIOS = {}


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return B.emul_lib(tmp_path_factory.mktemp("fft64_emul"))


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    for (path, n), (b, f) in sorted(RATIOS.items(), key=lambda kv: -kv[1][0])[:12]:
        print(f"worst ratio  path {path}  N {n:8d}  bin {b:.3f}  frame {f:.3f}")


def rnd(rng, n, scale=1.0):
    return scale * (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n))


def inputs(rng, n, frames=2):
    """random frames, exact-bin tones and tones whose samples carry one-signed relative jitter (the sums at the tone's
    bin grow to S_f, and every rounding sees operands of one sign)"""
    t = np.arange(n)
    k0 = int(rng.integers(0, n))
    tone = np.exp(2j * np.pi * ((k0 * t) % n) / n)
    jit = tone * (1.0 + rng.integers(1, 1 << 20, n) * 2.0 ** -52)
    return np.concatenate([rnd(rng, n * frames), tone, jit])


def run_check(emul, x, n, inverse, what):
    y = B.emulate(emul, x, n, inverse)
    return B.check(y, x, n, inverse, what, RATIOS)


# --------------------------------------------------------------------------------------------- the exact reference
@pytest.mark.parametrize("n", [3, 8, 17, 64])
def test_reference_matches_mpmath(n):
    mp = pytest.importorskip("mpmath")
    mp.mp.prec = 160
    rng = np.random.default_rng(n)
    x = rnd(rng, n)
    ref = B.exact(x, n, False)[0]
    s = np.abs(x).sum()
    for k in range(n):
        want = mp.fsum(mp.mpc(float(x[j].real), float(x[j].imag)) * mp.expjpi(-2 * mp.mpf(j * k % n) / n)
                       for j in range(n))
        got = mp.mpc(mp.mpf(float(ref[k].real)) + mp.mpf(float(ref[k].real - np.longdouble(float(ref[k].real)))),
                     mp.mpf(float(ref[k].imag)) + mp.mpf(float(ref[k].imag - np.longdouble(float(ref[k].imag)))))
        assert float(abs(got - want)) <= B.REF_TAU * s, (n, k)


# --------------------------------------------------------------------------------------------- emulation vs bound
@pytest.mark.parametrize("inverse", [0, 1])
@pytest.mark.parametrize("log2n", range(0, 21))
def test_every_power_of_two_meets_the_bound(emul, log2n, inverse):
    n = 1 << log2n
    rng = np.random.default_rng(100 + log2n)
    run_check(emul, inputs(rng, n, 2 if n < (1 << 18) else 1), n, inverse, f"pow2 {n}")


@pytest.mark.parametrize("inverse", [0, 1])
def test_every_length_up_to_300_meets_the_bound(emul, inverse):
    rng = np.random.default_rng(7)
    for n in range(1, 301):
        run_check(emul, inputs(rng, n), n, inverse, f"n {n}")


@pytest.mark.parametrize("inverse", [0, 1])
@pytest.mark.parametrize("n", [127, 128, 129, 4095, 4096, 4097, 8191, 8192, 8193, 1000, 48000, 65521, 65535, 65537,
                               (1 << 19) - 1, 1 << 19])
def test_path_boundaries_and_listed_lengths_meet_the_bound(emul, n, inverse):
    rng = np.random.default_rng(n)
    run_check(emul, inputs(rng, n, 1), n, inverse, f"n {n}")


@pytest.mark.parametrize("n", [1, 2, 3, 4, 8, 16, 100, 127, 128, 129, 256, 300, 1024, 4096])
def test_impulses_at_every_position_meet_the_bound(emul, n):
    x = np.zeros((n, n), np.complex128)
    x[np.arange(n), np.arange(n)] = 1.0 - 0.75j
    for inverse in (0, 1):
        run_check(emul, x.reshape(-1), n, inverse, f"impulses {n}")


@pytest.mark.parametrize("n", [16, 100, 1000, 8192])
def test_scaled_and_subnormal_frames_meet_the_bound(emul, n):
    rng = np.random.default_rng(n)
    base = rnd(rng, n)
    frames = [base * 2.0 ** 500, base * 2.0 ** -500, base * 2.0 ** -1060, np.full(n, 5e-324 + 5e-324j), base * 2.0 ** -1022]
    run_check(emul, np.concatenate(frames), n, 0, f"scaled {n}")


@pytest.mark.parametrize("n", [4, 16, 100, 1000, 8192])
def test_zero_and_non_finite_frames_stay_in_their_frame(emul, n):
    rng = np.random.default_rng(n)
    x = rnd(rng, 4 * n)
    x[:n] = 0.0
    x[n + n // 2] = np.inf
    x[2 * n + n // 3] = complex(np.nan, 0.0)
    y = B.emulate(emul, x, n)
    assert np.all(y[:n] == 0)
    B.check(y, x, n, False, f"edges {n}")  # frames 1 and 2 entirely non-finite, frame 3 within its bound


# --------------------------------------------------------------------------------------------- planted defects
def rejects(y, x, n, inverse, good):
    """the check a GPU result goes through: bit-identical to the emulation and within the bound"""
    return not B.same_bits(y, good) or bound_rejects(y, x, n, inverse)


def bound_rejects(y, x, n, inverse):
    try:
        B.check(y, x, n, inverse)
    except AssertionError:
        return True
    return False


@pytest.mark.parametrize("mutation,n,inverse", [
    (1, 4096, 0), (1, 1 << 16, 0),   # one twiddle at f32 precision
    (2, 64, 0), (2, 1000, 1),        # one bin off by 2^16 ulp
    (3, 48000, 0),                   # chirp angle without the integer reduction
    (5, 1000, 0),                    # NaN leaking into the next chirp-z frame
    (6, 4096, 1), (6, 1 << 14, 1),   # inverse plan with a forward twiddle in its last pass
])
def test_bound_rejects_each_planted_defect(emul, mutation, n, inverse):
    rng = np.random.default_rng(mutation)
    x = inputs(rng, n, 1)
    if mutation == 5:
        x[n // 2] = np.nan
    good = B.emulate(emul, x, n, inverse)
    bad = B.emulate(emul, x, n, inverse, mutation=mutation)
    assert rejects(bad, x, n, inverse, good)
    assert bound_rejects(bad, x, n, inverse), mutation


def test_f64_chirp_spectrum_is_rejected(emul):
    # the chirp spectrum from an f64 FFT: its error is of the order of the chirp-z bound itself, so the bits catch it
    n = 48000
    x = inputs(np.random.default_rng(4), n, 1)
    good = B.emulate(emul, x, n)
    bad = B.emulate(emul, x, n, mutation=4)
    assert rejects(bad, x, n, False, good)
    eb = np.abs(bad - good).max()
    assert eb > 0
    print(f"f64 chirp spectrum: max |diff| {eb:.3e}")


# ------------------------------------------------------------------------------------------------ header, build
def test_header_states_the_contract():
    h = open(os.path.join(ROOT, "include", "comms_b200.h")).read()
    sec = h[h.index("FFT over Complex<f64>"):h.index("CB_API int cb_fft_f64_run_dev")]
    for s in ("|X'[k] - X[k]| <= tau * S_f + floor", "||X' - X||_2 <= rho * ||X||_2 + sqrt(N) floor",
              "floor = 16 N 2^-1074 (chirp-z: 64 M sqrt(2N) 2^-1074)", "u = 2^-53",
              "powers of two (8 .. 4096):      tau = rho = 4 log2(N) u",
              "powers of two (8192 .. 2^20):   tau = rho = (4 log2(N) + 4) u",
              "direct sums (N <= 128):         tau = (3 N + 1) u,              rho = sqrt(N) tau",
              "tau = sqrt(2N - 1) (8 log2(M) + 12) u + 8 u,   rho = sqrt(2) tau",
              "Determinism.", "batch size", "split into calls", "cb_fft_f64_run vs cb_fft_f64_run_dev", "stream",
              "A zero frame gives exact zeros", "changes no\n * other frame", "CB_ERR_UNSUPPORTED", "2^19", "2^20"):
        assert s in sec, s


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
    hits = {k: v for k, v in usage.items() if "fft64_" in k}
    assert len(hits) == 6, sorted(hits)
    for name, (regs, stack) in hits.items():
        assert stack == 0, (name, stack)
        if "cols" in name:  # 512 threads per CTA (__launch_bounds__(512))
            assert regs * 512 <= 65536, (name, regs)


def test_cpp_node_compiles(tmp_path):
    src = tmp_path / "fft64_node.cpp"
    src.write_text('#include "comms_b200_nodes.hpp"\n'
                   "using namespace comms_b200;\n"
                   "void use() {\n"
                   "    FFTBatchNodeF64 a(1000, false);\n"
                   "    std::vector<c64> x(1000, c64{1.0, 0.0});\n"
                   "    auto r = a.run(x);\n"
                   "    (void)r;\n"
                   "}\n")
    subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(ROOT, "comms-rs_b200", "host"), str(src)], check=True)
