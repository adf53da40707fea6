"""Every bin of the Complex<f64> FFT (cb_fft_f64, FFTBatchNodeF64) against the CPU emulation of its paths
(tests/emul/fft_f64_emul.cpp): bit for bit, NaN positions compared as NaN, and within the header's per-bin and
per-frame bounds of the clongdouble reference (include/comms_b200.h).  Batches cross the two-step and chirp-z group
boundaries (GROUP_BYTES of work buffer per group) with special frames on both sides; calls split every way, host and
device entries, streams and error returns.  Needs a B200: `pytest -m gpu`.
"""
import itertools

import numpy as np
import pytest

import fft64_bounds as B

pytestmark = pytest.mark.gpu

GROUP_BYTES = 64 << 20
SIZES = [1, 2, 3, 4, 7, 8, 16, 64, 100, 127, 128, 129, 512, 1000, 1024, 4096, 4097, 8192, 48000, 65521, 65536,
         (1 << 19) - 1, 1 << 20]
RATIOS = {}


@pytest.fixture(scope="module")
def cb():
    import comms_rs_b200 as m

    m.init(0)
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t

    return t


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return B.emul_lib(tmp_path_factory.mktemp("fft64_emul"))


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    for (path, n), (b, f) in sorted(RATIOS.items()):
        print(f"worst ratio  path {path}  N {n:8d}  bin {b:.3f}  frame {f:.3f}")


def rnd(rng, n, scale=1.0):
    return scale * (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n))


def group_of(n):
    if B.path_of(n) == B.TWOSTEP:
        return max(1, GROUP_BYTES // (16 * n))
    if B.path_of(n) == B.CHIRPZ:
        return max(1, GROUP_BYTES // (16 * B.chirp_m(n)))
    return None


def run_dev(torch, node, x, stream=0):
    d_in = torch.from_numpy(np.ascontiguousarray(x).view(np.float64)).cuda()
    d_out = torch.empty_like(d_in)
    node.run_dev(d_in.data_ptr(), len(x), d_out.data_ptr(), stream)
    torch.cuda.synchronize()
    return d_out.cpu().numpy().view(np.complex128)


def frames_for(rng, n, g):
    """a batch crossing the first group boundary (when there is one) with zero, subnormal, 2^+-500, Inf and NaN frames
    on both sides"""
    nf = (g + 2) if g else 6
    nf = max(nf, 6)
    x = rnd(rng, n * nf)
    b = g if g and g < nf - 1 else nf // 2
    spec = {b - 1: "inf", b: "nan", b - 2 if b >= 2 else b + 2: "zero", b + 1: "sub"}
    for f, kind in spec.items():
        fr = x[f * n:(f + 1) * n]
        if kind == "inf":
            fr[n // 3] = np.inf
        elif kind == "nan":
            fr[0] = complex(0.0, np.nan)
        elif kind == "zero":
            fr[:] = 0.0
        else:
            fr[:] = fr * 2.0 ** -1060
    if nf > 4:
        x[:n] *= 2.0 ** 500
        x[(nf - 1) * n:] *= 2.0 ** -500
    return x


@pytest.mark.parametrize("inverse", [0, 1])
@pytest.mark.parametrize("n", SIZES)
def test_every_bin_matches_the_emulation_and_the_bound(cb, torch, emul, n, inverse):
    rng = np.random.default_rng(n + 7 * inverse)
    x = frames_for(rng, n, group_of(n))
    node = cb.FFTBatchNodeF64(n, bool(inverse))
    got = run_dev(torch, node, x)
    want = B.emulate(emul, x, n, inverse)
    assert B.same_bits(got, want), n
    B.check(got, x, n, inverse, f"n {n}", RATIOS)
    zero = ~np.any(x.reshape(-1, n), axis=1)
    assert np.all(got.reshape(-1, n)[zero] == 0)


@pytest.mark.parametrize("n", [16, 1000, 8192, 48000])
def test_split_calls_and_host_entry_give_the_same_bits(cb, torch, n):
    rng = np.random.default_rng(n)
    nf = 5
    x = rnd(rng, n * nf)
    node = cb.FFTBatchNodeF64(n)
    whole = run_dev(torch, node, x)
    assert B.same_bits(node.run(x), whole)
    for cuts in itertools.product([0, 1], repeat=nf - 1):  # every composition of the 5 frames into calls
        parts, start = [], 0
        for i, c in enumerate(cuts + (1,)):
            if c:
                parts.append(run_dev(torch, node, x[start * n:(i + 1) * n]))
                start = i + 1
        assert B.same_bits(np.concatenate(parts), whole), cuts
    s = cb.FFTSampleNodeF64(n)
    outs = [s.run(v) for v in x[:n]]
    assert all(o is None for o in outs[:-1]) and B.same_bits(outs[-1], whole[:n])


def test_error_returns(cb, torch):
    lib = cb._lib.load()
    import ctypes as C

    h = C.c_void_p()
    assert lib.cb_fft_f64_create(0, 0, C.byref(h)) == cb._lib.CB_ERR_INVALID_ARG
    for bad in ((1 << 20) + 1, 1 << 21, (1 << 19) + 1):
        assert lib.cb_fft_f64_create(bad, 0, C.byref(h)) == cb._lib.CB_ERR_UNSUPPORTED, bad
    node = cb.FFTBatchNodeF64(64)
    d = torch.zeros(2 * 64 * 4 + 2, dtype=torch.float64, device="cuda")
    p = d.data_ptr()
    with pytest.raises(cb.CbError):
        node.run_dev(p, 100, p + 16 * 128, 0)           # not a multiple of fft_size
    with pytest.raises(cb.CbError):
        node.run_dev(p + 8, 64, p + 16 * 128, 0)        # misaligned input
    with pytest.raises(cb.CbError):
        node.run_dev(p, 64, p + 16 * 128 + 8, 0)        # misaligned output
    with pytest.raises(cb.CbError):
        node.run_dev(p, 128, p + 16 * 64, 0)            # overlap
    with pytest.raises(cb.NodeError):
        node.run(np.zeros(65, np.complex128))           # the node's run() reports a DataError


def test_two_handles_on_two_streams_and_one_handle_on_two_streams(cb, torch, emul):
    rng = np.random.default_rng(3)
    n, nf = 48000, 40
    x = rnd(rng, n * nf)
    want = B.emulate(emul, x, n)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    a, b = cb.FFTBatchNodeF64(n), cb.FFTBatchNodeF64(n)
    d_in = torch.from_numpy(x.view(np.float64)).cuda()
    o1, o2, o3 = torch.empty_like(d_in), torch.empty_like(d_in), torch.empty_like(d_in)
    torch.cuda.synchronize()
    a.run_dev(d_in.data_ptr(), len(x), o1.data_ptr(), s1.cuda_stream)
    b.run_dev(d_in.data_ptr(), len(x), o2.data_ptr(), s2.cuda_stream)
    half = len(x) // 2
    a.run_dev(d_in.data_ptr(), half, o3.data_ptr(), s2.cuda_stream)
    a.run_dev(d_in.data_ptr() + 16 * half, half, o3.data_ptr() + 16 * half, s1.cuda_stream)
    torch.cuda.synchronize()
    for o in (o1, o2, o3):
        assert B.same_bits(o.cpu().numpy().view(np.complex128), want)


def test_one_large_call_on_sampled_frames(cb, torch, emul):
    n, total = 4096, 1 << 26
    g = torch.Generator(device="cuda").manual_seed(5)
    d_in = torch.rand(2 * total, dtype=torch.float64, device="cuda", generator=g) * 2 - 1
    d_out = torch.empty_like(d_in)
    node = cb.FFTBatchNodeF64(n)
    node.run_dev(d_in.data_ptr(), total, d_out.data_ptr(), 0)
    torch.cuda.synchronize()
    nf = total // n
    for f in [0, 1, nf // 3, nf // 2 + 1, nf - 2, nf - 1]:
        x = d_in[2 * n * f:2 * n * (f + 1)].cpu().numpy().view(np.complex128)
        got = d_out[2 * n * f:2 * n * (f + 1)].cpu().numpy().view(np.complex128)
        assert B.same_bits(got, B.emulate(emul, x, n)), f
        B.check(got, x, n, False, "large", RATIOS)
