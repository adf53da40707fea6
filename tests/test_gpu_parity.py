"""Parity of the CUDA path (through the C ABI) against the CPU oracle and the
reference's golden vectors.  Needs a B200: `pytest -m gpu`.

Tolerances (BASELINE.json north_star): FIR / mixer / polyphase complex-f32
relative L2 <= 1e-5; FFT relative L2 <= 1e-4; integer / index work bit-exact.
"""
import numpy as np
import pytest

from golden import reference_vectors as G

pytestmark = pytest.mark.gpu

FIR_TOL = 1e-5
FFT_TOL = 1e-4


@pytest.fixture(scope="module")
def cb():
    import comms_rs_b200 as m

    m.init(0)
    return m


def rel_l2(a, b):
    a = np.asarray(a).astype(np.complex128).ravel()
    b = np.asarray(b).astype(np.complex128).ravel()
    assert a.shape == b.shape, (a.shape, b.shape)
    d = np.linalg.norm(b)
    return np.linalg.norm(a - b) / d if d > 0 else np.linalg.norm(a - b)


def rnd_c32(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


# ------------------------------------------------------------------ FIR
def test_fir_golden_vector(cb):
    # src/filter/fir_node.rs:259-314: small integers are exact in f32 -> exact equality
    x = np.array([complex(*p) for p in G.FIR_INPUT], np.complex64)
    t = np.array([complex(*p) for p in G.FIR_TAPS], np.complex64)
    node = cb.FirNode(t)
    outs = [node.run(s) for s in x]
    assert [(int(v.real), int(v.imag)) for v in outs[:9]] == G.FIR_EXPECT
    node = cb.BatchFirNode(t)
    out = np.concatenate([node.run(x[i:i + 2]) for i in range(0, len(x), 2)])  # fir_node.rs:368-425
    assert [(int(v.real), int(v.imag)) for v in out] == G.BATCH_FIR_EXPECT


@pytest.mark.parametrize("ntaps", [1, 5, 16, 17, 32, 33, 63, 64, 65, 100, 128, 129, 200, 1024])
@pytest.mark.parametrize("cplx", [False, True])
def test_fir_matches_oracle(cb, oracle, ntaps, cplx):
    rng = np.random.default_rng(ntaps * 2 + cplx)
    n = 40_000 + ntaps
    x = rnd_c32(rng, n)
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    want, st = oracle.batch_fir(x, t, np.zeros(ntaps, np.complex64))
    node = cb.BatchFirNode(t)
    got = node.run(x)
    assert rel_l2(got, want) <= FIR_TOL
    assert node.state.tobytes() == st.tobytes()  # delay line is bit-exact (copies only)


@pytest.mark.parametrize("path", ["cuda", "auto", "tc"])
@pytest.mark.parametrize("sizes", [[0], [1], [1, 1, 1], [3, 0, 5], [255, 257, 4096, 1], [100_003, 7, 4097]])
def test_fir_batch_invariance_and_ragged(cb, oracle, sizes, path, monkeypatch):
    # path: COMMS_B200_FIR_PATH (read by cb_fir_create) -- CUDA-core kernels only, automatic choice,
    # or the tensor-core kernel for every batch size
    monkeypatch.setenv("COMMS_B200_FIR_PATH", path)
    rng = np.random.default_rng(11)
    t = rnd_c32(rng, 64)
    x = rnd_c32(rng, sum(sizes))
    want, st = oracle.batch_fir(x, t, np.zeros(64, np.complex64))
    node = cb.BatchFirNode(t)
    pos, outs = 0, []
    for s in sizes:
        outs.append(node.run(x[pos:pos + s]))
        assert len(outs[-1]) == s
        pos += s
    got = np.concatenate(outs) if outs else np.zeros(0, np.complex64)
    assert rel_l2(got, want) <= FIR_TOL if len(x) else True
    assert node.state.tobytes() == st.tobytes()
    one = cb.BatchFirNode(t).run(x)
    if path == "cuda":
        # CUDA-core kernels: one-shot result equals the batched one bit for bit
        assert one.tobytes() == got.tobytes()
    elif len(x):
        # tensor-core kernel: block-scaled split-fp16 products, batch edges visible only at the 1e-7 level
        assert rel_l2(one, got) <= 2e-6


@pytest.mark.parametrize("ntaps,nstate", [(64, 64), (33, 40), (40, 17), (5, 5), (8, 0), (64, 200)])
def test_fir_initial_state_and_zip_truncation(cb, oracle, ntaps, nstate):
    # BatchFirNode::new(taps, Some(state)); zip(taps, state) truncates (fir.rs:99)
    rng = np.random.default_rng(ntaps * 100 + nstate)
    t, s0, x = rnd_c32(rng, ntaps), rnd_c32(rng, nstate), rnd_c32(rng, 3000)
    want, st = oracle.batch_fir(x, t, s0)
    node = cb.BatchFirNode(t, s0)
    got = node.run(x)
    assert rel_l2(got, want) <= FIR_TOL
    assert node.state.tobytes() == st.tobytes()


def test_fir_state_get_set_resume(cb, oracle):
    rng = np.random.default_rng(5)
    t, x = rnd_c32(rng, 64), rnd_c32(rng, 10_000)
    a = cb.BatchFirNode(t)
    y1 = a.run(x[:6000])
    b = cb.BatchFirNode(t)
    b.state = a.state  # checkpoint / resume on another handle (segment + halo partitioning)
    y2 = b.run(x[6000:])
    want, _ = oracle.batch_fir(x, t, np.zeros(64, np.complex64))
    assert rel_l2(np.concatenate([y1, y2]), want) <= FIR_TOL


def test_fir_unaligned_host_pointers(cb, oracle):
    rng = np.random.default_rng(6)
    t = rnd_c32(rng, 64)
    buf = rnd_c32(rng, 5001)
    x = buf[1:]  # 8-byte aligned only
    want, _ = oracle.batch_fir(x, t, np.zeros(64, np.complex64))
    assert rel_l2(cb.BatchFirNode(t).run(x), want) <= FIR_TOL


# ------------------------------------------------------------------ resample
@pytest.mark.parametrize("data,rate,expect", G.DECIMATE_CASES)
def test_decimate_golden(cb, data, rate, expect):
    assert cb.DecimateNode(rate).run(np.array(data, np.int32)).tolist() == expect


@pytest.mark.parametrize("data,rate,expect", G.UPSAMPLE_CASES)
def test_upsample_golden(cb, data, rate, expect):
    assert cb.UpsampleNode(rate).run(np.array(data, np.int32)).tolist() == expect


@pytest.mark.parametrize("dtype", [np.uint8, np.int16, np.float32, np.complex64, np.complex128])
@pytest.mark.parametrize("rate", [0, 1, 2, 3, 10, 1000])
def test_resample_bit_exact(cb, oracle, dtype, rate):
    rng = np.random.default_rng(rate)
    a = rng.integers(0, 200, 10_001).astype(dtype)
    assert cb.DecimateNode(rate).run(a).tobytes() == oracle.decimate(a, rate).tobytes()
    b = a[:1000]
    assert cb.UpsampleNode(rate).run(b).tobytes() == oracle.upsample(b, rate).tobytes()
    assert len(cb.DecimateNode(rate).run(a[:0])) == 0


# ------------------------------------------------------------------ interp / decim fused
def test_pulse_golden_vector(cb):
    # src/pulse.rs:129-183: rect taps x4 -> each symbol repeated 4 times
    node = cb.PulseNode(np.ones(4, np.complex64), G.PULSE_SPS)
    out = np.concatenate([node.run(np.array([complex(*s)], np.complex64)) for s in G.PULSE_SYMBOLS])
    assert [(int(v.real), int(v.imag)) for v in out] == G.PULSE_EXPECT


@pytest.mark.parametrize("L,ntaps,cplx", [(4, 32, False), (2, 32, False), (8, 64, False), (8, 1024, False),
                                          (3, 17, False), (4, 32, True), (5, 100, True), (4, 30, False)])
def test_polyphase_interp_matches_upsample_then_fir(cb, oracle, L, ntaps, cplx):
    rng = np.random.default_rng(L * 1000 + ntaps)
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    sym = rnd_c32(rng, 20_011)
    st = np.zeros(ntaps, np.complex64)
    node = cb.BatchFirNode(t, None, decim=1, interp=L)
    pos, outs, wants = 0, [], []
    for s in (1, 4095, 10_000, 5915):
        w, st = oracle.batch_fir(oracle.upsample(sym[pos:pos + s], L), t, st)
        wants.append(w)
        outs.append(node.run(sym[pos:pos + s]))
        assert len(outs[-1]) == s * L  # sample counts are exact
        pos += s
    assert rel_l2(np.concatenate(outs), np.concatenate(wants)) <= FIR_TOL
    assert node.state.tobytes() == st.tobytes()


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("L,ntaps", [(8, 1024), (8, 64), (8, 1000), (8, 1), (8, 1100), (4, 32), (4, 30), (4, 400), (4, 3)])
def test_polyphase_tensor_core_path(cb, oracle, L, ntaps, cplx, monkeypatch):
    # K3-TC (fir_ptc_kernel.cu): the tcgen05 Toeplitz-GEMM polyphase bank, forced for every batch size,
    # against upsample -> batch_fir of the oracle (src/util/resample_node.rs:120-131 + src/filter/fir.rs:87-102)
    monkeypatch.setenv("COMMS_B200_FIR_PATH", "tc")
    rng = np.random.default_rng(L * 7000 + ntaps)
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    sizes = (1, 4095, 10_000, 5915, 2, 30_001)
    sym = rnd_c32(rng, sum(sizes))
    # per-tile block scaling: a quiet stretch and a loud stretch must both keep 1e-5
    sym[12_000:16_000] *= np.float32(1e-4)
    sym[30_000:34_000] *= np.float32(3e3)
    st = np.zeros(ntaps, np.complex64)
    node = cb.BatchFirNode(t, None, decim=1, interp=L)
    pos, outs, wants = 0, [], []
    for s in sizes:
        w, st = oracle.batch_fir(oracle.upsample(sym[pos:pos + s], L), t, st)
        wants.append(w)
        outs.append(node.run(sym[pos:pos + s]))
        assert len(outs[-1]) == s * L
        pos += s
    got, want = np.concatenate(outs), np.concatenate(wants)
    assert rel_l2(got, want) <= FIR_TOL
    # interior of the quiet stretch (its own tiles, after the filter has forgotten the louder past)
    lo, hi = (12_000 + 2 * ntaps // L + 4200) * L, 16_000 * L
    assert rel_l2(got[lo:hi], want[lo:hi]) <= FIR_TOL
    assert node.state.tobytes() == st.tobytes()
    monkeypatch.setenv("COMMS_B200_FIR_PATH", "cuda")
    ref = cb.BatchFirNode(t, None, decim=1, interp=L).run(sym)
    assert rel_l2(got, ref) <= 2e-6


@pytest.mark.parametrize("path", ["tc", "cuda"])
@pytest.mark.parametrize("L,ntaps,cplx", [(4, 32, False), (8, 1024, False), (8, 64, True), (1, 64, True), (3, 17, False)])
def test_fir_with_fused_i16_quantiser(cb, oracle, L, ntaps, cplx, path, monkeypatch):
    # filter -> `(8192.0 * x) as i16` -> interleaved i16 IQ (examples/single_thread_bpsk.rs:40-48, src/io/raw_iq.rs:185-223)
    # "tc": polyphase banks quantise inside the tcgen05 kernel's epilogue; "cuda": f32 scratch + quantiser kernel.
    monkeypatch.setenv("COMMS_B200_FIR_PATH", path)
    rng = np.random.default_rng(L * 31 + ntaps)
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    t = (t / np.float32(np.abs(t).sum() / 3)).astype(np.complex64)  # some outputs saturate at +-4
    x = rnd_c32(rng, 20_003)
    a, b = cb.BatchFirNode(t, None, interp=L), cb.BatchFirNode(t, None, interp=L)
    f32 = np.concatenate([b.run(x[:7]), b.run(x[7:])])
    peak = float(np.abs(f32.view(np.float32)).max())
    # large enough that some outputs saturate; a power of two (one fused multiply) or not (two roundings kept)
    scale = float(2.0 ** np.ceil(np.log2(50000.0 / peak))) if L != 8 else float(np.float32(50000.0 / peak))
    got = np.concatenate([a.run_i16(x[:7], scale), a.run_i16(x[7:], scale)])
    # identical to quantising the product's own f32 result (bit-exact integer stage) ...
    want_same = oracle.quantize_i16(f32, scale).reshape(-1, 2)
    assert got.shape == want_same.shape == (len(x) * L, 2)
    assert np.array_equal(got, want_same)
    # ... and within one LSB of the quantised oracle filter output (the f32 results differ by ~1e-7 relative)
    w, _ = oracle.batch_fir(oracle.upsample(x, L), t, np.zeros(ntaps, np.complex64))
    d = np.abs(got.astype(np.int32) - oracle.quantize_i16(w, scale).reshape(-1, 2).astype(np.int32))
    assert d.max() <= 1 and (d != 0).mean() < 2e-2
    assert (np.abs(got) == 32767).any() or (got == -32768).any()
    assert a.state.tobytes() == b.state.tobytes()


@pytest.mark.parametrize("D,ntaps,cplx", [(5, 63, False), (10, 63, False), (2, 64, True), (7, 33, True), (1000, 16, False)])
def test_decimating_fir_phase_resets_per_batch(cb, oracle, D, ntaps, cplx):
    # BatchFirNode -> DecimateNode: indices 0, D, 2D.. of EACH batch (resample_node.rs:53-65)
    rng = np.random.default_rng(D * 100 + ntaps)
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    x = rnd_c32(rng, 30_007)
    st = np.zeros(ntaps, np.complex64)
    node = cb.BatchFirNode(t, None, decim=D)
    pos = 0
    for s in (1, 13, 9999, 10_000, 9994):
        f, st = oracle.batch_fir(x[pos:pos + s], t, st)
        want = oracle.decimate(f, D)
        got = node.run(x[pos:pos + s])
        assert len(got) == len(want) == -(-s // D)
        assert rel_l2(got, want) <= FIR_TOL
        pos += s
    assert node.state.tobytes() == st.tobytes()


def test_interp_then_decim_rational(cb, oracle):
    rng = np.random.default_rng(77)
    t = rng.uniform(-1, 1, 48).astype(np.complex64)
    x = rnd_c32(rng, 5000)
    f, _ = oracle.batch_fir(oracle.upsample(x, 3), t, np.zeros(48, np.complex64))
    want = oracle.decimate(f, 2)
    got = cb.BatchFirNode(t, None, decim=2, interp=3).run(x)
    assert len(got) == len(want) and rel_l2(got, want) <= FIR_TOL


# ------------------------------------------------------------------ mixer
@pytest.mark.parametrize("phase,expect", [(None, G.MIXER_EXPECT_PHASE0), (0.1, G.MIXER_EXPECT_PHASE01)])
def test_mixer_golden_vector(cb, phase, expect):
    # src/mixer.rs:184-223, 274-313; f32 in/out here so the tolerance is f32 rounding of |y| ~ 10
    node = cb.MixerNode(G.MIXER_DPHASE, phase)
    got = np.array([node.run(np.complex64(v)) for v in G.MIXER_INPUT])
    assert np.all(np.abs(got - np.array(expect)) < 2e-6)
    node = cb.MixerNode(G.MIXER_DPHASE, phase)
    assert np.all(np.abs(node.run(np.array(G.MIXER_INPUT, np.complex64)) - np.array(expect)) < 2e-6)


@pytest.mark.parametrize("dphase", [0.123, -0.7, 6.0, 3 * 2 * np.pi + 0.25, 0.0])
def test_mixer_matches_oracle_and_carries_phase(cb, oracle, dphase):
    rng = np.random.default_rng(3)
    x = rnd_c32(rng, 200_001)
    ref = oracle.Mixer(0.2, dphase)
    node = cb.MixerNode(dphase, 0.2)
    assert node.dphase == ref.dphase
    pos = 0
    for s in (1, 2, 99_999, 100_000):
        want = ref.mix(x[pos:pos + s])
        got = node.run(x[pos:pos + s])
        assert rel_l2(got, want) <= FIR_TOL
        pos += s
    # phases agree modulo 2 pi (the oracle's single conditional wrap vs fmod)
    d = (node.phase - ref.phase) % (2 * np.pi)
    assert min(d, 2 * np.pi - d) < 1e-9


# ------------------------------------------------------------------ FFT
def test_fft10_golden_vector(cb):
    # src/fft/fft_node.rs:194-244 (batch) and :286-332 (sample node)
    x = np.array(G.FFT10_INPUT, np.complex64)
    got = cb.FFTBatchNode(10, False).run(x)
    assert np.all(np.abs(got - np.array(G.FFT10_EXPECT)) < G.FFT10_TOL)
    node = cb.FFTSampleNode(10, False)
    outs = [node.run(v) for v in x]
    assert all(o is None for o in outs[:-1])
    assert np.all(np.abs(outs[-1] - np.array(G.FFT10_EXPECT)) < G.FFT10_TOL)


@pytest.mark.parametrize("n", [1, 2, 3, 4, 8, 10, 12, 16, 32, 64, 100, 128, 256, 512, 1000, 1024, 2048, 4096, 8192,
                               16384, 32768, 65536, 1 << 17, 1 << 20,
                               # any other length (rustfft plans every size): direct up to 128, chirp-z beyond
                               127, 129, 255, 384, 1023, 4095, 4097, 5000, 10007, 48000, 65535, 100000, 300000])
@pytest.mark.parametrize("inverse", [False, True])
def test_fft_matches_oracle(cb, oracle, n, inverse):
    rng = np.random.default_rng(n + inverse)
    frames = 3 if n <= 65536 else (2 if n & (n - 1) else 1)
    x = rnd_c32(rng, frames * n)
    want = oracle.fft(x, n, inverse)
    got = cb.FFTBatchNode(n, inverse).run(x)
    assert rel_l2(got, want) <= FFT_TOL
    for f in range(frames):  # per frame too, so one bad frame cannot hide
        assert rel_l2(got[f * n:(f + 1) * n], want[f * n:(f + 1) * n]) <= FFT_TOL


@pytest.mark.parametrize("path", ["cluster", "cluster1", "cluster2", "cluster16", "twopass", "rows", "rows2", "big", "fourstep", "cpipe", "rowspf"])
@pytest.mark.parametrize("inverse", [False, True])
def test_fft65536_paths(cb, oracle, path, inverse, monkeypatch):
    # K5-C: one HBM pass on an 8-CTA cluster (distributed shared memory) vs the four-step fallback
    monkeypatch.setenv("COMMS_B200_FFT_PATH", path)
    rng = np.random.default_rng(65536 + inverse)
    n, frames = 65536, 5
    x = rnd_c32(rng, frames * n)
    x[2 * n:3 * n] = 0
    x[2 * n + 12345] = 1  # an impulse frame: every output has modulus 1 and a known phase
    want = oracle.fft(x, n, inverse)
    got = cb.FFTBatchNode(n, inverse).run(x)
    for f in range(frames):
        assert rel_l2(got[f * n:(f + 1) * n], want[f * n:(f + 1) * n]) <= FFT_TOL


@pytest.mark.parametrize("frames", [1, 2, 3, 19, 75])
def test_fft65536_pipelined_cluster_frame_counts(cb, oracle, frames, monkeypatch):
    # K5-P (fft_cpipe_kernel.cu): persistent clusters, frames round-robin over the resident clusters; fewer frames than
    # clusters, exactly one or two per cluster (the pipeline's prologue / epilogue iterations) and several per cluster
    monkeypatch.setenv("COMMS_B200_FFT_PATH", "cpipe")
    n = 65536
    rng = np.random.default_rng(frames)
    x = rnd_c32(rng, frames * n)
    for inverse in (False, True):
        got = cb.FFTBatchNode(n, inverse).run(x)
        for f in sorted({0, frames // 2, frames - 1}):
            want = oracle.fft(x[f * n:(f + 1) * n], n, inverse)
            assert rel_l2(got[f * n:(f + 1) * n], want) <= FFT_TOL, (f, inverse)
        e_in = (np.abs(x.reshape(frames, n).astype(np.complex128)) ** 2).sum(axis=1)
        e_out = (np.abs(got.reshape(frames, n).astype(np.complex128)) ** 2).sum(axis=1)
        assert np.all(np.abs(e_out / (n * e_in) - 1) < 1e-5)  # every frame: Parseval


@pytest.mark.parametrize("n", [16, 32, 64, 128])
def test_fft_small_sizes_many_frames(cb, oracle, n, monkeypatch):
    # 16 .. 128 points (fft2_small_frames_kernel):
    # a CTA moves 4096 contiguous points through shared memory; frame
    # counts that fill CTAs exactly, leave a ragged last CTA, or are smaller than one CTA; forward and inverse; device
    # buffers that are only 8-byte aligned (scalar accesses instead of 16-byte ones) give the same bits
    import os
    import torch

    rng = np.random.default_rng(n)
    per_cta = 4096 // n
    for frames in (1, per_cta - 1, per_cta, per_cta + 1, 5 * per_cta + 3, 40 * per_cta):
        x = rnd_c32(rng, frames * n)
        for inverse in (False, True):
            got = cb.FFTBatchNode(n, inverse).run(x)
            want = oracle.fft(x, n, inverse)
            assert rel_l2(got, want) <= FFT_TOL, (frames, inverse)
            for f in sorted({0, frames // 2, frames - 1}):
                assert rel_l2(got[f * n:(f + 1) * n], want[f * n:(f + 1) * n]) <= FFT_TOL, (frames, inverse, f)
    frames = 3 * per_cta + 5
    x = rnd_c32(rng, frames * n)
    d = torch.zeros(frames * n + 1, dtype=torch.complex64, device="cuda")
    d[1:] = torch.from_numpy(x).cuda()
    o = torch.zeros(frames * n + 2, dtype=torch.complex64, device="cuda")
    node = cb.FFTBatchNode(n, False)
    node.run_dev(d.data_ptr() + 8, frames * n, o.data_ptr() + 8, 0)  # both pointers 8 mod 16
    torch.cuda.synchronize()
    res = o.cpu().numpy()
    assert res[0] == 0 and res[-1] == 0
    assert res[1:-1].tobytes() == node.run(x).tobytes()


@pytest.mark.parametrize("n", [8192, 16384])
def test_fft_8192_16384_two_level_kernel(cb, oracle, n, monkeypatch):
    # fft2_two_level_kernel: 256 x 32 / 256 x 64 inside one CTA (rows by half-warps, columns by 2 / 4 adjacent threads);
    # several frame counts, both directions, 8-byte aligned device buffers (scalar loads), and agreement with the
    # generic radix-16 kernel (the default)
    import torch

    monkeypatch.setenv("COMMS_B200_FFT_8K16K", "two")  # not the default: the generic kernel measured faster
    rng = np.random.default_rng(n + 5)
    for frames in (1, 5, 37):
        x = rnd_c32(rng, frames * n)
        x[(frames // 2) * n:(frames // 2 + 1) * n] = 0
        x[(frames // 2) * n + 4321] = 1  # an impulse frame: every output has modulus 1 and a known phase
        for inverse in (False, True):
            got = cb.FFTBatchNode(n, inverse).run(x)
            for f in sorted({0, frames // 2, frames - 1}):
                want = oracle.fft(x[f * n:(f + 1) * n], n, inverse)
                assert rel_l2(got[f * n:(f + 1) * n], want) <= FFT_TOL, (frames, inverse, f)
    frames = 7
    x = rnd_c32(rng, frames * n)
    node = cb.FFTBatchNode(n, False)
    ref = node.run(x)
    d = torch.zeros(frames * n + 1, dtype=torch.complex64, device="cuda")
    d[1:] = torch.from_numpy(x).cuda()
    o = torch.zeros(frames * n + 2, dtype=torch.complex64, device="cuda")
    node.run_dev(d.data_ptr() + 8, frames * n, o.data_ptr() + 8, 0)
    torch.cuda.synchronize()
    res = o.cpu().numpy()
    assert res[0] == 0 and res[-1] == 0 and res[1:-1].tobytes() == ref.tobytes()
    monkeypatch.setenv("COMMS_B200_FFT_8K16K", "generic")
    assert rel_l2(cb.FFTBatchNode(n, False).run(x), ref) <= 2e-6


@pytest.mark.parametrize("path", ["rows", "rowspf"])
@pytest.mark.parametrize("frames", [1, 2, 17, 40, 150, 700])
def test_fft65536_ring_frame_counts(cb, oracle, frames, path, monkeypatch):
    # K5-R / K5-R2 (fft_rows_kernel.cu): persistent kernels over tickets with the intermediate in a ring of 96 frames;
    # fewer frames than the lag, more than the ring (slots reused, both dependency directions exercised), and enough
    # for every CTA to run many items back to back (the prefetching form's steady state)
    monkeypatch.setenv("COMMS_B200_FFT_PATH", path)
    n = 65536
    rng = np.random.default_rng(1000 + frames)
    x = rnd_c32(rng, frames * n)
    for inverse in (False, True):
        got = cb.FFTBatchNode(n, inverse).run(x)
        for f in sorted({0, frames // 3, frames // 2, frames - 1}):
            want = oracle.fft(x[f * n:(f + 1) * n], n, inverse)
            assert rel_l2(got[f * n:(f + 1) * n], want) <= FFT_TOL, (f, inverse)
        e_in = (np.abs(x.reshape(frames, n).astype(np.complex128)) ** 2).sum(axis=1)
        e_out = (np.abs(got.reshape(frames, n).astype(np.complex128)) ** 2).sum(axis=1)
        assert np.all(np.abs(e_out / (n * e_in) - 1) < 1e-5)  # every frame: Parseval
    if frames >= 150:  # a repeated run of the same handle gives the same bits (no dependence on who won which ticket)
        node = cb.FFTBatchNode(n, False)
        a, b = node.run(x), node.run(x)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("n", [1024, 4096, 65536])
def test_fft_roundtrip_and_linearity(cb, n):
    rng = np.random.default_rng(n)
    x, y = rnd_c32(rng, 4 * n), rnd_c32(rng, 4 * n)
    f, b = cb.FFTBatchNode(n, False), cb.FFTBatchNode(n, True)
    assert rel_l2(b.run(f.run(x)) / n, x) <= FFT_TOL  # unnormalised both ways
    assert rel_l2(f.run(x + 2 * y), f.run(x) + 2 * f.run(y)) <= FFT_TOL
    imp = np.zeros(n, np.complex64)
    imp[1] = 1
    k = np.arange(n)
    assert rel_l2(f.run(imp), np.exp(-2j * np.pi * k / n)) <= FFT_TOL  # sign convention
    assert rel_l2(b.run(imp), np.exp(+2j * np.pi * k / n)) <= FFT_TOL


def test_fft_wrong_length_is_data_error(cb):
    node = cb.FFTBatchNode(1024, False)
    with pytest.raises(cb.NodeError) as e:
        node.run(np.zeros(1000, np.complex64))
    assert e.value.kind == cb.NodeError.DataError
    with pytest.raises(cb.CbError):
        cb.FFTBatchNode(0, False)


# ------------------------------------------------------------------ FM demod
def test_fm_demod_matches_oracle(cb, oracle):
    rng = np.random.default_rng(9)
    x = rnd_c32(rng, 100_000)
    x[0] = -1 - 1j  # first output is atan2(-0, -0) = pi (SURVEY appendix A)
    ref, node = oracle.FM(), cb.FMDemodNode()
    for a, b in ((0, 1), (1, 50_000), (50_000, 100_000)):
        want, got = ref.demod(x[a:b]), node.run(x[a:b])
        # the product is formed with the same individually rounded ops; atan2f may differ by an ulp
        d = np.abs(got.astype(np.float64) - want.astype(np.float64))
        d = np.minimum(d, 2 * np.pi - d)
        assert d.max() < 1e-6
    assert cb.FMDemodNode().run(np.array([-1 - 1j], np.complex64))[0] == np.float32(np.pi)
    assert cb.FMDemodNode().run(np.array([1 + 1j], np.complex64))[0] == 0.0


# ------------------------------------------------------------------ fused bank (BASELINE cfg 4)
FM_RADIO_TAPS_N = 63


def _lowpass(n):
    k = np.arange(n) - (n - 1) / 2
    return (np.sinc(k / 5) * np.hamming(n) / 5).astype(np.float32).astype(np.complex64)


@pytest.mark.parametrize("mix,fm,cplx,D", [(True, True, False, 10), (True, False, False, 10), (False, True, False, 5),
                                           (False, False, True, 4), (True, True, True, 3), (True, True, False, 1)])
def test_chain_bank_matches_node_chain(cb, oracle, mix, fm, cplx, D):
    rng = np.random.default_rng(D)
    C, taps = 7, _lowpass(FM_RADIO_TAPS_N)
    if cplx:
        taps = (taps * np.exp(1j * 0.1 * np.arange(len(taps)))).astype(np.complex64)
    dph = -2 * np.pi * rng.uniform(-0.4, 0.4, C)
    ph0 = rng.uniform(0, 6, C)
    bank = cb.ChainBank(C, taps, D, dphase=dph if mix else None, phase=ph0 if mix else None, with_fm=fm)
    refs = [oracle.FmChain(dph[c], ph0[c], taps, D, do_mix=mix, do_fm=fm) for c in range(C)]
    for n in (1, 131_072 // 8, 9_999, 20_003, 40_000, 131_072):
        x = rnd_c32(rng, C * n).reshape(C, n)
        got = bank.run(x)
        assert got.shape == (C, -(-n // D))  # bit-exact sample counts, phase restarts per call
        for c in range(C):
            want = refs[c].run(x[c])
            if fm:
                d = np.abs(got[c].astype(np.float64) - want.astype(np.float64))
                d = np.minimum(d, 2 * np.pi - d)
                # angle error ~ |dy| / |y|: tiny everywhere except where |y| itself is ~0
                assert np.median(d) < 2e-6 and np.mean(d > 1e-3) < 2e-3, (c, n, np.median(d), d.max())
            else:
                assert rel_l2(got[c], want) <= FIR_TOL, (c, n)


@pytest.mark.parametrize("mix,fm,D,n", [(False, True, 5, 131_072), (True, True, 10, 131_072), (True, False, 10, 40_000),
                                        (False, True, 5, 9_999), (True, True, 4, 16_384)])
def test_chain_bank_u8_input_fused_convert(cb, oracle, mix, fm, D, n):
    # fm_radio as shipped: RTL-SDR bytes -> ConvertNode (x - 127.5) / 127.5 -> FIR -> /D -> FM (examples/fm_radio.rs:84-87,144-164)
    # D in {5, 10} with n % 8 == 0 converts inside the TMA-staged kernel; other shapes convert into a scratch first.
    import torch

    rng = np.random.default_rng(D * 7 + n)
    C, taps = 5, _lowpass(FM_RADIO_TAPS_N)
    dph = -2 * np.pi * rng.uniform(-0.4, 0.4, C)
    a = cb.ChainBank(C, taps, D, dphase=dph if mix else None, with_fm=fm)
    b = cb.ChainBank(C, taps, D, dphase=dph if mix else None, with_fm=fm)
    refs = [oracle.FmChain(dph[c], 0.0, taps, D, do_mix=mix, do_fm=fm) for c in range(C)]
    for call in range(3):  # state (history, phase, FM prev) carried across calls
        iq = rng.integers(0, 256, (C, n, 2), dtype=np.uint8)
        # stand-alone converter: bit-exact against the oracle's ((x as f32) - 127.5) / 127.5
        d8 = torch.from_numpy(iq.reshape(-1)).cuda()
        df = torch.empty(C * n, dtype=torch.complex64, device="cuda")
        ts = torch.cuda.Stream()
        torch.cuda.synchronize()
        cb.convert_u8_dev(d8.data_ptr(), C * n, df.data_ptr(), ts.cuda_stream)
        torch.cuda.synchronize()
        xf = df.cpu().numpy().reshape(C, n)
        assert xf.view(np.float32).tobytes() == oracle.u8_to_f32(iq.reshape(-1)).tobytes()
        got = a.run_u8(iq)
        same = b.run(xf)
        assert got.shape == same.shape == (C, -(-n // D))
        if D in (5, 10) and n % 8 == 0:
            # fused kernel: the span holds b - 127.5 (exact) and ConvertNode's division sits in the taps -- the same
            # algebra as convert-then-filter, different rounding points
            if fm:
                dd = np.abs(got.astype(np.float64) - same.astype(np.float64))
                dd = np.minimum(dd, 2 * np.pi - dd)
                assert np.median(dd) < 1e-6 and np.mean(dd > 1e-3) < 2e-3
            else:
                assert rel_l2(got, same) <= 1e-6
        else:  # other shapes convert into a scratch first: the very same f32 values reach the filter
            assert got.tobytes() == same.tobytes()
        for c in range(C):
            want = refs[c].run(xf[c])
            if fm:
                d = np.abs(got[c].astype(np.float64) - want.astype(np.float64))
                d = np.minimum(d, 2 * np.pi - d)
                assert np.median(d) < 2e-6 and np.mean(d > 1e-3) < 2e-3, (c, call)
            else:
                assert rel_l2(got[c], want) <= FIR_TOL, (c, call)


@pytest.mark.parametrize("fm", [True, False])
@pytest.mark.parametrize("ntaps,n", [(63, 131_072), (63, 40_000), (64, 10_240 * 2 + 8), (17, 10_240 * 3 - 40), (5, 2_048), (63, 8)])
def test_chain_bank_u8_tensor_core_path(cb, oracle, fm, ntaps, n, monkeypatch):
    # K2-TC (chain_tc_kernel.cu): bytes -> ConvertNode -> <= 64 real taps -> /5 [-> FM] as five polyphase Toeplitz GEMMs on
    # tcgen05, forced for every batch size; against convert-then-filter of the product's CUDA-core kernel and the oracle
    # chain (examples/fm_radio.rs:84-97,144-160).  Tiles of 2048 outputs: batch lengths below, at and across tile edges.
    monkeypatch.setenv("COMMS_B200_CHAIN_PATH", "tc")
    rng = np.random.default_rng(ntaps * 13 + n)
    C, taps = 3, _lowpass(ntaps)
    a = cb.ChainBank(C, taps, 5, dphase=None, with_fm=fm)
    refs = [oracle.FmChain(0.0, 0.0, taps, 5, do_mix=False, do_fm=fm) for _ in range(C)]
    for call in range(3):  # history and FM state carried across calls; the decimation phase restarts with each
        iq = rng.integers(0, 256, (C, n, 2), dtype=np.uint8)
        if call == 1:
            iq[0, : n // 2] = 128  # a constant stretch: outputs near the filter's DC response, angles near 0 / pi
        got = a.run_u8(iq)
        xf = oracle.u8_to_f32(iq.reshape(-1)).view(np.complex64).reshape(C, n)
        assert got.shape == (C, -(-n // 5))
        for c in range(C):
            want = refs[c].run(xf[c])
            if fm:
                d = np.abs(got[c].astype(np.float64) - want.astype(np.float64))
                d = np.minimum(d, 2 * np.pi - d)
                assert np.median(d) < 2e-6 and np.mean(d > 1e-3) < 5e-3, (c, call, np.median(d), d.max())
            else:
                assert rel_l2(got[c], want) <= FIR_TOL, (c, call, rel_l2(got[c], want))
    monkeypatch.setenv("COMMS_B200_CHAIN_PATH", "v3")
    b = cb.ChainBank(C, taps, 5, dphase=None, with_fm=False)
    monkeypatch.setenv("COMMS_B200_CHAIN_PATH", "tc")
    t = cb.ChainBank(C, taps, 5, dphase=None, with_fm=False)
    iq = rng.integers(0, 256, (C, n, 2), dtype=np.uint8)
    y_tc = t.run_u8(iq)
    monkeypatch.setenv("COMMS_B200_CHAIN_PATH", "v3")
    y_cc = b.run_u8(iq)
    assert rel_l2(y_tc, y_cc) <= 1e-6  # the two kernel families agree far inside the tolerance


@pytest.mark.parametrize("decim,ntaps", [(5, 63), (10, 63), (2, 64), (4, 17), (8, 33), (5, 1), (3, 63), (1, 40), (5, 100)])
def test_real_input_fir_matches_oracle(cb, oracle, decim, ntaps):
    # Convert2Node -> filt2 -> Convert3Node -> dec2 (examples/fm_radio.rs:98-164) as one call: real samples in, real
    # parts out.  Fused kernel for <= 64 taps and D in {2,4,5,8,10}; the other shapes run widen + complex filter + .re
    rng = np.random.default_rng(decim * 1000 + ntaps)
    taps = _lowpass(ntaps) if ntaps > 1 else np.array([0.75], np.complex64)
    node = cb.BatchFirNode(taps, None, decim=decim)
    st = np.zeros(len(taps), np.complex64)
    # batch lengths around the 1024-output tile, odd lengths, a batch shorter than the filter
    for n in (1024 * decim, 1024 * decim + 1, 7, 26_215, 3 * 1024 * decim - 1, 1, 50_001):
        x = rng.uniform(-1, 1, n).astype(np.float32)
        got = node.run_real(x)
        full, st = oracle.batch_fir(x.astype(np.complex64), taps, st)
        want = oracle.decimate(full.real.astype(np.float32), decim)
        assert got.shape == want.shape
        assert rel_l2(got, want) <= FIR_TOL, (n, rel_l2(got, want))
    # the carried state is the reference's (Complex(x, 0), newest first)
    assert node.state.tobytes() == st.tobytes()
    # device entry with input and output that are only 4-byte aligned (scalar load / store paths)
    import torch

    n = 3 * 1024 * decim + 5
    x = rng.uniform(-1, 1, n).astype(np.float32)
    d_x = torch.zeros(n + 1, dtype=torch.float32, device="cuda")
    d_x[1:] = torch.from_numpy(x).cuda()
    no = -(-n // decim)
    d_y = torch.zeros(no + 1, dtype=torch.float32, device="cuda")
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()
    assert node.run_dev_real(d_x.data_ptr() + 4, n, d_y.data_ptr() + 4, no, ts.cuda_stream) == no
    torch.cuda.synchronize()
    full, st = oracle.batch_fir(x.astype(np.complex64), taps, st)
    assert rel_l2(d_y[1:].cpu().numpy(), oracle.decimate(full.real.astype(np.float32), decim)) <= FIR_TOL
    assert float(d_y[0]) == 0.0


def test_fm_radio_example_graph_on_device(cb, oracle):
    # examples/fm_radio.rs:144-164, the whole shipped graph with every hop on the GPU:
    #   bytes -> ConvertNode -> filt1 -> dec1(5) -> FMDemodNode -> Convert2Node -> filt2 -> Convert3Node -> dec2(5)
    # batches of 131072 IQ samples (262144 bytes, fm_radio.rs:144), state carried by filt1, fm and filt2
    import torch

    rng = np.random.default_rng(144)
    taps = _lowpass(FM_RADIO_TAPS_N)
    nb, n1 = 131_072, -(-131_072 // 5)
    n2 = -(-n1 // 5)
    front = cb.ChainBank(1, taps, 5, dphase=None, with_fm=True)   # convert + filt1 + dec1 + fm fused
    filt2 = cb.BatchFirNode(taps, None, decim=5)                   # filt2 + dec2 fused (decimation commutes with .re)
    ref_front = oracle.FmChain(0.0, 0.0, taps, 5, do_mix=False, do_fm=True)
    st2 = np.zeros(len(taps), np.complex64)
    ts = torch.cuda.Stream()
    s = ts.cuda_stream
    d_fm = torch.empty(n1, dtype=torch.float32, device="cuda")
    d_c = torch.empty(n1, dtype=torch.complex64, device="cuda")
    d_f2 = torch.empty(n2, dtype=torch.complex64, device="cuda")
    d_audio = torch.empty(n2, dtype=torch.float32, device="cuda")
    for batch in range(3):
        iq = rng.integers(0, 256, (nb, 2), dtype=np.uint8)
        d_iq = torch.from_numpy(iq.reshape(-1)).cuda()
        torch.cuda.synchronize()
        assert front.run_dev_u8(d_iq.data_ptr(), nb, d_fm.data_ptr(), n1, s) == n1
        if batch == 1:  # the same hops as separate device entries (Convert2Node / Convert3Node glue)
            cb.real_to_complex_dev(d_fm.data_ptr(), n1, d_c.data_ptr(), s)
            assert filt2.run_dev(d_c.data_ptr(), n1, d_f2.data_ptr(), n2, s) == n2
            cb.complex_real_dev(d_f2.data_ptr(), n2, d_audio.data_ptr(), s)
        else:           # Convert2Node -> filt2 -> Convert3Node -> dec2 as one kernel
            assert filt2.run_dev_real(d_fm.data_ptr(), n1, d_audio.data_ptr(), n2, s) == n2
        torch.cuda.synchronize()
        x = oracle.u8_to_f32(iq.reshape(-1)).view(np.complex64)
        fm_ref = ref_front.run(x)
        f2, st2 = oracle.batch_fir(fm_ref.astype(np.complex64), taps, st2)
        audio_ref = oracle.decimate(f2.real.astype(np.float32), 5)
        got = d_audio.cpu().numpy()
        assert got.shape == audio_ref.shape == (n2,)
        # angles wrap at +-pi: a 1e-7 difference there becomes 2 pi in the demodulated sample; compare the bulk
        d = np.abs(got.astype(np.float64) - audio_ref.astype(np.float64))
        assert np.median(d) < 5e-6 and np.mean(d > 1e-2) < 5e-3, (batch, np.median(d), d.max())


def _shaped_qpsk_f64(oracle, rng, nsym, sps, ntaps, alpha):
    sym = np.exp(1j * (2 * np.pi * rng.integers(0, 4, nsym) / 4 + np.pi / 4))
    up = np.zeros(nsym * sps, np.complex128)
    up[::sps] = sym
    taps = oracle.rrc_taps(ntaps, float(sps), alpha, dtype=np.complex128)
    out, _ = oracle.batch_fir(up, taps, np.zeros(ntaps, np.complex128))
    return out


@pytest.mark.parametrize("n,d,alpha,nsym,drop", [(10, 5, 0.5, 1000, 2), (2, 5, 0.25, 3000, 0), (4, 8, 0.35, 5000, 1),
                                                 (8, 0, 0.5, 100, 0), (3, 2, 1.0, 50, 0)])
def test_timing_estimator_matches_oracle(cb, oracle, n, d, alpha, nsym, drop):
    # TimingEstimator::push (src/demodulation/timing_estimator.rs:85-112): f64; the product sums in a tree, the
    # reference in index order: 1e-9 samples
    rng = np.random.default_rng(n * 100 + d)
    x = _shaped_qpsk_f64(oracle, rng, nsym, n, 10 * n + 1, alpha)[drop:]
    x = x + 0.01 * (rng.standard_normal(len(x)) + 1j * rng.standard_normal(len(x)))
    want = oracle.TimingEstimator(n, d, alpha).push(x)
    est = cb.TimingEstimator(n, d, alpha)
    got = est.push(x)
    assert abs(got - want) < 1e-9, (got, want)
    assert est.push(x) == got  # fixed reduction order: same bits every time
    if (n, d) == (10, 5):
        assert abs(drop + got) < 0.01  # the reference's own test (timing_estimator.rs:183-196)
    import torch

    d_x = torch.from_numpy(x).cuda()
    assert est.push_dev(d_x.data_ptr(), len(x)) == got
    assert est.push(x[:0]) == 0.0
    # fewer samples than the delay N*D + 1: every dout is a zero and the sum is exactly zero.  The reference then
    # returns the argument of a SIGNED zero (0 or -+N/2, decided by the signs of the first samples); the product
    # returns 0 (DESIGN.md, K7)
    if d == 0:
        assert abs(est.push(x[:1]) - oracle.TimingEstimator(n, d, alpha).push(x[:1])) < 1e-12
    else:
        assert est.push(x[:n * d]) == 0.0
        k = n * d + 1  # the first length with a non-zero term
        assert abs(est.push(x[:k]) - oracle.TimingEstimator(n, d, alpha).push(x[:k])) < 1e-9
    np.testing.assert_array_equal(cb.qfilt_taps(2 * n * d + 1, alpha, n), oracle.qfilt_taps(2 * n * d + 1, alpha, n))
    with pytest.raises(ValueError):
        cb.TimingEstimator(n, d, 1.5)


def test_timing_estimator_longest_filter(cb, oracle):
    # 2 N D + 1 = 4097 taps: the largest shared-memory tile; one more symbol of delay is refused
    n, d, alpha = 8, 256, 0.3
    rng = np.random.default_rng(4097)
    x = _shaped_qpsk_f64(oracle, rng, 2000, n, 10 * n + 1, alpha)
    want = oracle.TimingEstimator(n, d, alpha).push(x)
    assert abs(cb.TimingEstimator(n, d, alpha).push(x) - want) < 1e-9
    with pytest.raises(cb.CbError):
        cb.TimingEstimator(n, d + 1, alpha)


def test_frequency_estimator_matches_oracle(cb, oracle):
    # frequency_offset_estimate (src/demodulation/frequency_estimator.rs:27-42) and its test (:56-100)
    rng = np.random.default_rng(7)
    truth = 0.123456789
    x = _shaped_qpsk_f64(oracle, rng, 4096, 4, 16, 0.75)
    x = x * np.exp(1j * truth * np.arange(len(x)))
    want = oracle.frequency_offset_estimate(x)
    got = cb.frequency_offset_estimate(x)
    assert abs(got - want) < 1e-12 and abs(truth - got) < 0.01
    for m in (0, 1, 2, 3, 255, 256, 257, 2049):
        assert abs(cb.frequency_offset_estimate(x[:m]) - oracle.frequency_offset_estimate(x[:m])) < 1e-12, m
    import torch

    # a long pure tone on the device: the estimate is the tone's frequency whatever the length
    nbig = (1 << 24) + 5
    t = torch.arange(nbig, dtype=torch.float64, device="cuda") * (-0.3)
    d_x = torch.polar(torch.ones_like(t), t)
    assert abs(cb.frequency_offset_estimate_dev(d_x.data_ptr(), nbig) + 0.3) < 1e-9


def test_convert_i16_bit_exact(cb):
    import torch

    v = np.array([0, 1, -1, 32767, -32768, 8192, -12345, 77], dtype=np.int16)
    d = torch.from_numpy(v).cuda()
    out = torch.empty(len(v), dtype=torch.float32, device="cuda")
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()
    cb.convert_i16_dev(d.data_ptr(), len(v) // 2, 1.0, out.data_ptr(), ts.cuda_stream)
    torch.cuda.synchronize()
    assert out.cpu().numpy().tobytes() == v.astype(np.float32).tobytes()
    cb.convert_i16_dev(d.data_ptr(), len(v) // 2, 1.0 / 8192.0, out.data_ptr(), ts.cuda_stream)
    torch.cuda.synchronize()
    assert out.cpu().numpy().tobytes() == (v.astype(np.float32) * np.float32(1.0 / 8192.0)).tobytes()


# ------------------------------------------------------------------ BASELINE cfg 1 (single_thread_bpsk)
@pytest.mark.parametrize("nsym", [1 << 16, 1 << 20])  # 2^20 symbols in 256 batches of 4096: the config as specified
def test_bpsk_chain_config1(cb, oracle, nsym):
    import torch

    batch, sps = 4096, 4
    bits_ref, shaped_ref, iq_ref, st_ref = oracle.bpsk_chain(nsym, batch=batch, sps=sps)
    bits, _ = cb.prn_bits(0xB8, 0x01, nsym, 8)
    assert bits.tobytes() == bits_ref.tobytes()  # PRN bits: bit-exact
    taps = oracle.rrc_taps(32, 4.0, 0.25)
    fir = cb.BatchFirNode(taps, None, interp=sps)
    dev = torch.device("cuda:0")
    # one explicit stream for the whole chain: stream 0 would mean "the handle's own stream" to the FIR node
    # but the legacy default stream to the stateless stages, and the two do not order against each other
    ts = torch.cuda.Stream()
    s = ts.cuda_stream
    d_bits = torch.from_numpy(bits).to(dev)
    torch.cuda.synchronize()
    d_sym = torch.empty(nsym, dtype=torch.complex64, device=dev)
    d_shaped = torch.empty(nsym * sps, dtype=torch.complex64, device=dev)
    d_iq = torch.empty(nsym * sps * 2, dtype=torch.int16, device=dev)
    assert cb.bits_to_symbols_dev(d_bits.data_ptr(), nsym, 0, d_sym.data_ptr(), s) == nsym
    for b in range(0, nsym, batch):  # state carried across batches (single_thread_bpsk.rs:19,39)
        m = fir.run_dev(d_sym.data_ptr() + 8 * b, batch, d_shaped.data_ptr() + 8 * b * sps, batch * sps, s)
        assert m == batch * sps
    cb.quantize_i16_dev(d_shaped.data_ptr(), nsym * sps * 2, 8192.0, d_iq.data_ptr(), s)
    torch.cuda.synchronize()
    sym = d_sym.cpu().numpy()
    assert sym.tobytes() == oracle.example_bpsk_map(bits_ref).tobytes()  # symbol map: bit-exact
    shaped = d_shaped.cpu().numpy()
    assert rel_l2(shaped, shaped_ref) <= FIR_TOL
    assert fir.state.tobytes() == st_ref.tobytes()
    # quantiser itself is bit-exact on identical input
    assert d_iq.cpu().numpy().tobytes() == oracle.quantize_i16(shaped).tobytes()
    # and end to end the i16 stream differs from the reference chain by at most 1 LSB, rarely
    diff = np.abs(d_iq.cpu().numpy().astype(np.int32) - iq_ref.astype(np.int32))
    assert diff.max() <= 1 and (diff != 0).mean() < 1e-2


def test_qpsk_symbol_map_bit_exact(cb, oracle):
    import torch

    bits, _ = cb.prn_bits(0xB8, 0x01, 20_000, 8)
    d_bits = torch.from_numpy(bits).cuda()
    d_sym = torch.empty(10_000, dtype=torch.complex64, device="cuda")
    assert cb.bits_to_symbols_dev(d_bits.data_ptr(), 20_000, 1, d_sym.data_ptr(), torch.cuda.current_stream().cuda_stream) == 10_000
    torch.cuda.synchronize()
    assert d_sym.cpu().numpy().tobytes() == oracle.example_qpsk_map(bits).tobytes()
    assert cb.prn_bits(0xC0, 0x01, 128, 8)[0].tolist() == G.PRN_C0_01  # src/prns.rs:211-220


# ------------------------------------------------------------------ full-size properties (BASELINE cfg 2 / 3)
def test_fir_full_size_windows_and_properties(cb, oracle):
    """2^28-sample stream resident on the device: random interior windows against the
    oracle (seeded with the preceding K samples as state), batch invariance, linearity."""
    import torch

    n, K, seed = 1 << 28, 64, 1234
    s = torch.cuda.current_stream().cuda_stream
    x = torch.empty(n, dtype=torch.complex64, device="cuda")
    y = torch.empty(n, dtype=torch.complex64, device="cuda")
    cb.synth_uniform_dev(seed, 0, n, x.data_ptr(), s)
    taps_r = oracle.rrc_taps(64, 4.0, 0.25)
    taps_c = (taps_r * np.exp(1j * 0.1 * np.arange(64))).astype(np.complex64)
    for taps in (taps_r, taps_c):
        node = cb.BatchFirNode(taps)
        assert node.run_dev(x.data_ptr(), n, y.data_ptr(), n, s) == n
        torch.cuda.synchronize()
        rng = np.random.default_rng(1)
        starts = [0, n - 5000] + [int(v) for v in rng.integers(K, n - 5000, 6)]
        for st in starts:
            lo = max(st - K, 0)
            xin = oracle.synth_uniform_c32(seed, lo, st - lo + 5000)
            assert xin.tobytes() == x[lo:st + 5000].cpu().numpy().tobytes()  # generator parity, bit-exact
            state = np.zeros(K, np.complex64)
            state[: st - lo] = xin[: st - lo][::-1]
            want, _ = oracle.batch_fir(xin[st - lo:], taps, state)
            assert rel_l2(y[st:st + 5000].cpu().numpy(), want) <= FIR_TOL
        # 256 batches of 2^20 with carried state == one shot, bit for bit
        y2 = torch.empty(n, dtype=torch.complex64, device="cuda")
        node2 = cb.BatchFirNode(taps)
        B = 1 << 20
        for b in range(0, n, B):
            node2.run_dev(x.data_ptr() + 8 * b, B, y2.data_ptr() + 8 * b, B, s)
        torch.cuda.synchronize()
        if not torch.equal(y.view(torch.float32), y2.view(torch.float32)):  # say where: tile, offset, batch
            bad = torch.nonzero((y.view(torch.int32) != y2.view(torch.int32)).view(-1, 2).any(dim=1)).flatten()
            tiles = torch.unique(bad // 4096)
            raise AssertionError(f"batched != one shot: {bad.numel()} samples in {tiles.numel()} tiles, first tiles {tiles[:8].tolist()} "
                                 f"(tile % 256: {(tiles[:8] % 256).tolist()}), offsets in tile {(bad[:8] % 4096).tolist()}, "
                                 f"values {y[int(bad[0])].item()} vs {y2[int(bad[0])].item()}")
        assert node.state.tobytes() == node2.state.tobytes()
        del y2
    # impulse response: x = delta at 1000 -> y[1000 + k] = h[k]
    x.zero_()
    x[1000] = 1
    node = cb.BatchFirNode(taps_c)
    node.run_dev(x.data_ptr(), 1 << 20, y.data_ptr(), 1 << 20, s)
    torch.cuda.synchronize()
    # (tensor-core path: taps travel as two fp16 terms, 22 bits -- not bit-exact, but far inside FIR_TOL)
    assert rel_l2(y[1000:1064].cpu().numpy(), taps_c) <= 1e-6
    assert float(y[:1000].abs().max()) == 0.0 and float(y[1064:1 << 20].abs().max()) == 0.0


@pytest.mark.parametrize("n", [1024, 4096, 65536])
def test_fft_full_size_roundtrip(cb, oracle, n):
    import torch

    total, seed = 1 << 28, 99
    s = torch.cuda.current_stream().cuda_stream
    x = torch.empty(total, dtype=torch.complex64, device="cuda")
    f = torch.empty(total, dtype=torch.complex64, device="cuda")
    cb.synth_uniform_dev(seed, 0, total, x.data_ptr(), s)
    fwd, inv = cb.FFTBatchNode(n, False), cb.FFTBatchNode(n, True)
    fwd.run_dev(x.data_ptr(), total, f.data_ptr(), s)
    torch.cuda.synchronize()
    rng = np.random.default_rng(n)
    for fr in [0, total // n - 1] + [int(v) for v in rng.integers(0, total // n, 4)]:
        xin = oracle.synth_uniform_c32(seed, fr * n, n)
        assert rel_l2(f[fr * n:(fr + 1) * n].cpu().numpy(), oracle.fft(xin, n, False)) <= FFT_TOL
    # Parseval as a checksum over the whole job: sum|X|^2 = N sum|x|^2
    ex = float((x.view(torch.float32).double() ** 2).sum())
    ef = float((f.view(torch.float32).double() ** 2).sum())
    assert abs(ef / (n * ex) - 1) < 1e-5
    back = torch.empty(total, dtype=torch.complex64, device="cuda")
    inv.run_dev(f.data_ptr(), total, back.data_ptr(), s)
    torch.cuda.synchronize()
    err = (back.view(torch.float32) / n - x.view(torch.float32)).double().norm() / x.view(torch.float32).double().norm()
    assert float(err) <= FFT_TOL


def test_comm_gather_single_rank(cb):
    # cb_comm_* / cb_gather_segments_dev (ncclAllGather bound by dlopen): with one rank the gather is the identity;
    # the 2-rank form is scripts/mg_gather_check.py (torchrun, one process per GPU)
    import torch

    g = cb.sharding.SegmentGather(1, 0, cb.sharding.SegmentGather.unique_id())
    x = torch.randn(2 * 10_000, device="cuda")
    y = torch.zeros_like(x)
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()
    g.gather_dev(x.data_ptr(), 10_000, y.data_ptr(), ts.cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(x, y)
    g.close()


def test_comm_single_rank_root_and_var_gather(cb):
    # the variable-length forms with one rank: a device copy into place (root) / the identity (all ranks)
    import torch

    g = cb.sharding.SegmentGather(1, 0, cb.sharding.SegmentGather.unique_id())
    x = torch.randn(2 * 4099, device="cuda")
    y, z = torch.zeros_like(x), torch.zeros_like(x)
    ts = torch.cuda.Stream()
    torch.cuda.synchronize()
    g.gather_to_root_dev(x.data_ptr(), [4099], 8, 0, y.data_ptr(), ts.cuda_stream)
    g.allgather_var_dev(x.data_ptr(), [4099], 8, z.data_ptr(), ts.cuda_stream)
    g.gather_to_root_dev(0, [0], 8, 0, 0, ts.cuda_stream)  # empty segment: a no-op, not a hang
    torch.cuda.synchronize()
    assert torch.equal(x, y) and torch.equal(x, z)
    with pytest.raises(cb.CbError):
        g.gather_to_root_dev(x.data_ptr(), [4099], 8, 3, y.data_ptr(), ts.cuda_stream)  # root out of range
    g.close()


def test_in_place_run_dev_is_rejected(cb):
    # include/comms_b200.h: input and output ranges of a *_run_dev call must not overlap (the kernels read neighbouring
    # tiles and rebuild the carried state from the input) -> CB_ERR_INVALID_ARG, state untouched
    import torch

    n = 1 << 14
    x = torch.randn(2 * n, device="cuda")
    y = torch.empty(2 * n, device="cuda")
    taps = np.ones(8, np.complex64)
    fir = cb.BatchFirNode(taps)
    st0 = fir.state.copy()
    for dst in (x.data_ptr(), x.data_ptr() + 8 * (n - 1), x.data_ptr() - 8 * (n - 1)):
        with pytest.raises(cb.CbError) as e:
            fir.run_dev(x.data_ptr(), n, dst, n, 0)
        assert e.value.status == cb._lib.CB_ERR_INVALID_ARG and "overlap" in str(e.value)
    assert fir.state.tobytes() == st0.tobytes()
    fir.run_dev(x.data_ptr(), n, y.data_ptr(), n, 0)  # disjoint: fine
    with pytest.raises(cb.CbError):
        cb.FMDemodNode().run_dev(x.data_ptr(), n, x.data_ptr(), 0)
    with pytest.raises(cb.CbError):
        cb.FFTBatchNode(1024).run_dev(x.data_ptr(), n, x.data_ptr() + 8 * 1024, 0)
    with pytest.raises(cb.CbError):
        cb.ChainBank(2, taps, 2, dphase=[0.1, 0.2]).run_dev(x.data_ptr(), n // 2, x.data_ptr(), n // 4, 0)
    with pytest.raises(cb.CbError):
        cb.BatchFirNode(taps, None, decim=5).run_dev_real(x.data_ptr(), n, x.data_ptr() + 64, n, 0)
    m = cb.MixerNode(0.1)
    m.run_dev(x.data_ptr(), n, x.data_ptr(), 0)  # element-wise: in place is allowed
    torch.cuda.synchronize()


def test_handle_state_is_ordered_across_streams(cb):
    # a handle used on two caller streams back to back (the Rust GpuBatchFirDevNode / C++ mirror pattern): the second
    # launch must see the history the first one is still writing, get_state must wait for both
    import oracle
    import torch

    rng = np.random.default_rng(11)
    taps = rnd_c32(rng, 48)
    n1, n2 = 1 << 22, 300
    xh = rnd_c32(rng, n1 + n2)
    want, st = oracle.batch_fir(xh[-4096:], taps, xh[-4096 - 48:-4096][::-1].copy())
    x = torch.from_numpy(xh).cuda()
    y = torch.empty_like(x)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(3):
        node = cb.BatchFirNode(taps)
        node.run_dev(x.data_ptr(), n1, y.data_ptr(), n1, sa.cuda_stream)
        node.run_dev(x.data_ptr() + 8 * n1, n2, y.data_ptr() + 8 * n1, n2, sb.cuda_stream)
        state = node.state  # cb_fir_get_state: waits for the last use on any stream
        assert state.tobytes() == st.tobytes()
        torch.cuda.synchronize()
        assert rel_l2(y[-4096:].cpu().numpy(), want) <= FIR_TOL
    # two 65536-point transforms on different streams share the handle's scratch ring and counters
    f = cb.FFTBatchNode(65536)
    xf = torch.from_numpy(rnd_c32(rng, 8 * 65536)).cuda()
    o1, o2, o3 = torch.empty_like(xf), torch.empty_like(xf), torch.empty_like(xf)
    torch.cuda.synchronize()
    f.run_dev(xf.data_ptr(), xf.numel(), o3.data_ptr(), sa.cuda_stream)
    torch.cuda.synchronize()
    f.run_dev(xf.data_ptr(), xf.numel(), o1.data_ptr(), sa.cuda_stream)
    f.run_dev(xf.data_ptr(), xf.numel(), o2.data_ptr(), sb.cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(torch.view_as_real(o1), torch.view_as_real(o3)) and torch.equal(torch.view_as_real(o2), torch.view_as_real(o3))


def test_large_pageable_host_call_is_staged_and_correct(cb):
    # a Rust Vec is pageable memory: host-pointer calls stage each chunk through pinned slots (the parallel copier above
    # 1 MiB; api.cu HostPipe::h2d / d2h); results must equal the pinned-buffer call bit for bit
    import ctypes as C
    import oracle
    import torch

    rng = np.random.default_rng(3)
    n = (1 << 22) * 2 + 12345  # three chunks of the 2-lane pipeline, ragged tail
    x = rnd_c32(rng, n)
    taps = rnd_c32(rng, 64)
    got = cb.BatchFirNode(taps).run(x)  # numpy memory: pageable
    xp = torch.from_numpy(x).pin_memory()
    yp = torch.empty(n, dtype=torch.complex64).pin_memory()
    node = cb.BatchFirNode(taps)
    cb._lib.check(cb.load().cb_fir_run(node._h, xp.data_ptr(), n, yp.data_ptr(), n, None))
    assert got.tobytes() == yp.numpy().tobytes()
    lo = (1 << 22) - 500
    want, _ = oracle.batch_fir(x[lo:lo + 1000], taps, x[lo - 64:lo][::-1].copy())
    assert rel_l2(got[lo:lo + 1000], want) <= FIR_TOL
    nf = (n // 4096) * 4096
    gf = cb.FFTBatchNode(4096).run(x[:nf])
    fp = torch.empty(nf, dtype=torch.complex64).pin_memory()
    f = cb.FFTBatchNode(4096)
    cb._lib.check(cb.load().cb_fft_run(f._h, xp.data_ptr(), nf, fp.data_ptr()))
    assert gf.tobytes() == fp.numpy().tobytes()
    gm = cb.MixerNode(0.37, 0.5).run(x)
    mp = torch.empty(n, dtype=torch.complex64).pin_memory()
    m = cb.MixerNode(0.37, 0.5)
    cb._lib.check(cb.load().cb_mixer_run(m._h, xp.data_ptr(), n, mp.data_ptr()))
    assert gm.tobytes() == mp.numpy().tobytes()


@pytest.mark.parametrize("interp,decim", [(1, 1), (4, 1), (1, 5)])
def test_small_host_calls_run_over_pinned_host_memory(cb, oracle, interp, decim):
    # cb_fir_run with input + output below 1 MiB: one kernel over pinned host memory, no copy engine (api.cu
    # ZEROCOPY_MAX_BYTES) -- the caller's buffers in place when they are pinned, the handle's slots when pageable.
    # Messages of both kinds, and one above the threshold (copy-engine path), interleaved on one handle: the carried
    # state lives on the device across all of them, so the stream must equal one oracle pass over the concatenation.
    import torch

    rng = np.random.default_rng(50 + interp + decim)
    taps = rnd_c32(rng, 64) if interp == 1 else rng.uniform(-1, 1, 32).astype(np.complex64)
    sizes = [4096, 4095, 200_000, 1, 4096 * 5, 63, 8190]
    sizes = [n - n % decim if n >= decim else decim for n in sizes]  # whole decimation periods: one oracle pass compares
    x = rnd_c32(rng, sum(sizes))
    node = cb.BatchFirNode(taps, None, interp=interp, decim=decim)
    outs, pos = [], 0
    for i, n in enumerate(sizes):
        seg = x[pos:pos + n]
        no = n * interp // decim
        if i % 2 == 0:
            outs.append(node.run(seg))  # numpy memory: pageable
        else:
            xp = torch.from_numpy(seg.copy()).pin_memory()
            yp = torch.empty(max(no, 1), dtype=torch.complex64).pin_memory()
            cb._lib.check(cb.load().cb_fir_run(node._h, xp.data_ptr(), n, yp.data_ptr(), max(no, 1), None))
            outs.append(yp.numpy()[:no].copy())
        assert len(outs[-1]) == no
        pos += n
    got = np.concatenate(outs)
    want, _ = oracle.batch_fir(oracle.upsample(x, interp) if interp > 1 else x, taps, np.zeros(len(taps), np.complex64))
    assert rel_l2(got, want[::decim]) <= FIR_TOL
    one = cb.BatchFirNode(taps, None, interp=interp, decim=decim).run(x)  # a single large call: copy-engine or TC path
    assert rel_l2(got, one) <= FIR_TOL
    if interp == 1 and decim == 1:
        # a pinned buffer used as input AND output of a small host call: not run over host memory in place (the kernel
        # would read samples it has already overwritten) but through the copy path, which tolerates it
        buf = torch.from_numpy(x[:4096].copy()).pin_memory()
        a, b = cb.BatchFirNode(taps), cb.BatchFirNode(taps)
        cb._lib.check(cb.load().cb_fir_run(a._h, buf.data_ptr(), 4096, buf.data_ptr(), 4096, None))
        assert buf.numpy().tobytes() == b.run(x[:4096]).tobytes()


def test_cpp_graph_message_rate_bench_runs(cb):
    """comms-rs_b200/host/bench_graph.cpp at small message counts: thread-per-node graphs with pooled device edges must
    deliver every message, and the device-edge cfg-1 graph must equal the host-edge graph bit for bit."""
    import json
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    host = os.path.join(root, "comms-rs_b200", "host")
    subprocess.run(["make", "-C", host, "-s", "all"], check=True)
    r = subprocess.run([os.path.join(host, "bench_graph"), "512", "48"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "bench_graph ok" in r.stdout
    lines = [json.loads(ln) for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 3 and lines[1]["bit_identical_to_host_edges"] is True
    assert lines[1]["pool_device"]["hits"] > 0  # blocks are recycled, not cudaMalloc'ed per message


# ------------------------------------------------------------------ i16 IQ on both edges (src/io/raw_iq.rs)
@pytest.mark.parametrize("ntaps,interp,decim,n", [(64, 1, 1, 300_000), (32, 4, 1, 70_000), (63, 1, 5, 100_003), (17, 3, 2, 5_001),
                                                   (64, 1, 1, (1 << 23) + 4099)])
def test_fir_iq16_edges_equal_the_separate_nodes(cb, oracle, ntaps, interp, decim, n):
    # cb_fir_run_iq16: IQBatchInput's i16 samples -> cast -> filter -> `(scale * y) as i16` (IQBatchOutput), 4 bytes per
    # sample on every edge; must equal convert -> cb_fir_run -> quantise bit for bit (small batches: one chunk; the
    # last case: three chunks of the 2-lane host pipeline with re-sent halos) and match the oracle chain
    rng = np.random.default_rng(ntaps * 100 + interp)
    t = rng.uniform(-1, 1, ntaps).astype(np.complex64) if interp > 1 or decim > 1 else rnd_c32(rng, ntaps)
    iq = rng.integers(-32768, 32768, size=(n, 2), dtype=np.int16)
    in_scale, out_scale = 1.0 / 32768.0, 3000.0
    x = (iq.astype(np.float32) * np.float32(in_scale)).view(np.complex64).ravel()
    a, b = cb.BatchFirNode(t, None, decim=decim, interp=interp), cb.BatchFirNode(t, None, decim=decim, interp=interp)
    cut = n // 3
    got = np.concatenate([a.run_iq16(iq[:cut], in_scale, out_scale), a.run_iq16(iq[cut:], in_scale, out_scale)])
    f32 = np.concatenate([b.run(x[:cut]), b.run(x[cut:])])
    assert np.array_equal(got, oracle.quantize_i16(f32, out_scale).reshape(-1, 2))
    assert a.state.tobytes() == b.state.tobytes()
    if n <= 300_000:
        st, parts = np.zeros(ntaps, np.complex64), []
        for seg in (x[:cut], x[cut:]):  # per call: the decimation phase restarts with every batch (resample_node.rs:53-65)
            w, st = oracle.batch_fir(oracle.upsample(seg, interp) if interp > 1 else seg, t, st)
            parts.append(oracle.decimate(w, decim) if decim > 1 else w)
        want = oracle.quantize_i16(np.concatenate(parts), out_scale).reshape(-1, 2)
        d = np.abs(got.astype(np.int32) - want.astype(np.int32))
        assert d.max() <= 1 and (d != 0).mean() < 2e-2  # same values up to the filter's rounding: rarely one LSB apart


def test_fir_iq16_device_call_alignments_and_tails(cb, oracle):
    # cb_fir_run_dev_iq16 on the tensor-core path (fir_tc_kernel IQ16): output buffers that are only 4-byte aligned take
    # the single-word stores, inputs that are not 16-byte aligned fall back to cast -> filter -> quantise, batch lengths
    # that are not multiples of four leave up to three samples to the converters -- all must give the same words
    import torch

    rng = np.random.default_rng(77)
    taps = rnd_c32(rng, 64)
    n = 262_144 + 3
    iq = rng.integers(-32768, 32768, size=(n + 8, 2), dtype=np.int16)
    d_iq = torch.from_numpy(iq).cuda()
    d_out = torch.zeros((n + 16, 2), dtype=torch.int16, device="cuda")
    in_scale, out_scale = 1.0 / 32768.0, 5000.0
    x = (iq.astype(np.float32) * np.float32(in_scale)).view(np.complex64).ravel()
    results = {}
    for in_off, out_off, m in ((0, 0, n), (0, 1, n), (0, 3, n - 1), (1, 0, n), (4, 8, n - 2), (0, 0, n - 3)):
        node = cb.BatchFirNode(taps)
        node.state = rnd_c32(np.random.default_rng(5), 64)  # a non-zero history: the first tile's halo is f32, not i16
        d_out.zero_()
        got_n = node.run_dev_iq16(d_iq.data_ptr() + 4 * in_off, m, in_scale, out_scale, d_out.data_ptr() + 4 * out_off, m, 0)
        torch.cuda.synchronize()
        assert got_n == m
        out = d_out.cpu().numpy()
        assert not out[:out_off].any() and not out[out_off + m:].any()  # nothing outside the output range
        ref = cb.BatchFirNode(taps)
        ref.state = rnd_c32(np.random.default_rng(5), 64)
        want = oracle.quantize_i16(ref.run(x[in_off:in_off + m]), out_scale).reshape(-1, 2)
        d = np.abs(out[out_off:out_off + m].astype(np.int32) - want.astype(np.int32))
        # aligned input: the fused kernel, bit-identical to quantising the f32 tensor-core result; the fall-back is
        # identical as well (same three steps)
        assert d.max() == 0, (in_off, out_off, m, int(d.max()))
        assert node.state.tobytes() == ref.state.tobytes()


def test_fft_iq16_input_equals_cast_then_fft(cb):
    rng = np.random.default_rng(9)
    iq = rng.integers(-32768, 32768, size=(8 * 4096, 2), dtype=np.int16)
    x = iq.astype(np.float32).view(np.complex64).ravel()
    f = cb.FFTBatchNode(4096)
    assert f.run_iq16(iq).tobytes() == f.run(x).tobytes()
    f2 = cb.FFTBatchNode(65536)
    iq2 = rng.integers(-2000, 2000, size=(3 * 65536, 2), dtype=np.int16)
    assert f2.run_iq16(iq2, 0.5).tobytes() == f2.run((iq2.astype(np.float32) * np.float32(0.5)).view(np.complex64).ravel()).tobytes()
    with pytest.raises(cb.NodeError):
        f.run_iq16(iq[:100])  # wrong length -> DataError, like the f32 entry
    # every kind of plan: single-kernel sizes and 65536 points read the i16 samples in their first pass (fft_kernels.cu
    # fft2_frames_iq16_kernel, fft_rows_kernel.cu IN16), the others widen first; all equal cast -> transform bit for bit
    for n, frames, inverse in ((16, 700, False), (64, 33, True), (1024, 9, False), (8192, 3, True), (16384, 5, False),
                               (32768, 3, False), (65536, 120, True), (1 << 17, 2, False), (1000, 7, False), (100, 3, True)):
        iq3 = rng.integers(-32768, 32768, size=(frames * n, 2), dtype=np.int16)
        sc = np.float32(1.0 / 1024)
        node = cb.FFTBatchNode(n, inverse)
        want = node.run((iq3.astype(np.float32) * sc).view(np.complex64).ravel())
        assert node.run_iq16(iq3, float(sc)).tobytes() == want.tobytes(), (n, inverse)
        import torch
        d_iq = torch.from_numpy(iq3).cuda()
        d_out = torch.empty(frames * n, dtype=torch.complex64, device="cuda")
        node.run_dev_iq16(d_iq.data_ptr(), frames * n, float(sc), d_out.data_ptr(), 0)
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes() == want.tobytes(), (n, inverse, "dev")


# ------------------------------------------------------------------ buffer pool (back-pressure for unbounded channels)
def test_buffer_pool_reuse_and_back_pressure(cb):
    # cb_buf_alloc_* come from a size-classed pool (no cudaMalloc / cudaFree per message); with a high-water mark the
    # source-side gate cb_pool_throttle blocks until a consumer releases (src/node/mod.rs:152: unbounded channels)
    import ctypes as C
    import threading
    import time

    lib = cb.load()
    for dev in (True, False):
        alloc = lib.cb_buf_alloc_device if dev else lib.cb_buf_alloc_pinned
        s0 = cb.pool_stats(dev)
        a = C.c_void_p()
        cb._lib.check(alloc(100_000, C.byref(a)))
        pa = lib.cb_buf_ptr(a)
        assert lib.cb_buf_bytes(a) == 100_000
        lib.cb_buf_release(a)
        b = C.c_void_p()
        cb._lib.check(alloc(120_000, C.byref(b)))  # same size class (128 KiB): the block comes back from the pool
        assert lib.cb_buf_ptr(b) == pa
        s1 = cb.pool_stats(dev)
        assert s1["hits"] == s0["hits"] + 1 and s1["live_bytes"] == s0["live_bytes"] + (1 << 17)
        lib.cb_buf_release(b)
        # high-water mark of three 1 MiB blocks: allocations never block, the gate is cb_pool_throttle (called by sources)
        cb.pool_configure(dev, max_live_bytes=s0["live_bytes"] + (3 << 20), timeout_ms=300)
        try:
            held = []
            for _ in range(4):
                h = C.c_void_p()
                cb._lib.check(alloc(1 << 20, C.byref(h)))
                held.append(h)
            t0 = time.perf_counter()
            rc = lib.cb_pool_throttle(0)  # nobody releases: fails after the configured timeout instead of hanging
            assert rc == cb._lib.CB_ERR_OOM and time.perf_counter() - t0 >= 0.25
            assert b"high-water" in lib.cb_last_error()
            threading.Timer(0.1, lambda: lib.cb_buf_release(held.pop())).start()  # a consumer drops its message
            t0 = time.perf_counter()
            cb._lib.check(lib.cb_pool_throttle(2000))  # blocks ~0.1 s, then proceeds
            assert 0.05 <= time.perf_counter() - t0 < 1.0
            cb._lib.check(lib.cb_pool_throttle(0))  # under the mark: returns at once
            assert cb.pool_stats(dev)["waits"] >= s0["waits"] + 2
            for h in held:
                lib.cb_buf_release(h)
        finally:
            cb.pool_configure(dev)
        assert cb.pool_stats(dev)["live_bytes"] == s0["live_bytes"]
    lib.cb_pool_trim()
    assert cb.pool_stats(True)["cached_bytes"] == 0


def test_pooled_buffer_waits_for_previous_owner(cb):
    # a block released while a kernel still reads it (consumer recorded `done` behind its launch) must not reach its
    # next owner before that kernel finished: the second owner overwrites it at once, the first result must not change
    import ctypes as C
    import torch

    lib = cb.load()
    n = 1 << 24
    x = torch.randn(2 * n, device="cuda")
    want = torch.empty(2 * n, device="cuda")
    m = cb.MixerNode(0.3)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    m.run_dev(x.data_ptr(), n, want.data_ptr(), sa.cuda_stream)
    torch.cuda.synchronize()
    for _ in range(3):
        buf = C.c_void_p()
        cb._lib.check(lib.cb_buf_alloc_device(8 * n, C.byref(buf)))
        p = lib.cb_buf_ptr(buf)
        cb._lib.check(lib.cb_decimate_dev(x.data_ptr(), n, 8, 1, p, n, None, sa.cuda_stream))  # producer fills the message
        cb._lib.check(lib.cb_buf_record_ready(buf, sa.cuda_stream))
        out = torch.empty(2 * n, device="cuda")
        torch.cuda.synchronize()
        m.phase = 0.0
        cb._lib.check(lib.cb_buf_wait_ready(buf, sb.cuda_stream))
        m.run_dev(p, n, out.data_ptr(), sb.cuda_stream)  # consumer reads it asynchronously ...
        cb._lib.check(lib.cb_buf_record_done(buf, sb.cuda_stream))
        lib.cb_buf_release(buf)  # ... and drops it at once
        nxt = C.c_void_p()
        cb._lib.check(lib.cb_buf_alloc_device(8 * n, C.byref(nxt)))  # same block, next owner
        assert lib.cb_buf_ptr(nxt) == p
        cb._lib.check(lib.cb_synth_uniform_dev(1, 0, n, p, sa.cuda_stream))  # overwrites immediately on another stream
        torch.cuda.synchronize()
        assert torch.equal(out, want)
        lib.cb_buf_release(nxt)


# ------------------------------------------------------------------ NCO batching shim (SURVEY 8(f) rank 4)
def test_nco_batch_matches_reference_recurrence(cb):
    # Nco::push (src/demodulation/nco.rs:71-77) applied in order; the product evaluates the same phases as a scan.
    # Truth = the recurrence in extended precision (phase mod 2 pi is all that reaches the output).  Tolerance: the
    # oracle's own f64 recurrence drifts by up to ~n * ulp(2 pi); the scan must be at least that close to the truth.
    import oracle

    rng = np.random.default_rng(5)
    for n, dphase, phase0, amp in ((1, 0.1, np.pi / 4, 0.01), (1000, 0.1, np.pi / 4, 0.01), (8191, 6.2, 0.0, 0.3),
                                   (1 << 20, 0.123456789, 1.0, 1e-3), (70001, -0.7, 3.0, 0.05)):
        perr = rng.uniform(-amp, amp, n)
        want = oracle.Nco(phase0, dphase).push(perr)
        node = cb.NcoNode(dphase, phase0)
        got = node.run(perr)
        dw = np.float64(oracle.Nco(phase0, dphase).dphase)
        assert node.dphase == dw
        ph = np.longdouble(phase0) + np.cumsum(np.longdouble(dw) + perr.astype(np.longdouble))
        truth = np.exp(1j * (ph % (2 * np.longdouble(np.pi) + np.longdouble(1.2246467991473532e-16) * 2)).astype(np.float64))
        e_orc = np.abs(want - truth).max()
        e_gpu = np.abs(got - truth).max()
        assert e_gpu <= max(2e-13, 2 * e_orc), (n, e_gpu, e_orc)
        assert np.abs(got - want).max() <= 1e-12 + 2e-16 * n * 8, (n, np.abs(got - want).max())
        # carried phase: continuing in a second batch equals one long batch
        node2 = cb.NcoNode(dphase, phase0)
        h = n // 3
        again = np.concatenate([node2.run(perr[:h]), node2.run(perr[h:])]) if h else got
        assert np.abs(again - got).max() <= 1e-12
        assert 0.0 <= node.phase < 2 * np.pi
        assert abs(np.exp(1j * node.phase) - got[-1]) <= 1e-12
    # one sample per call: the reference's NcoNode::run(f64)
    node, orc = cb.NcoNode(0.1, None), oracle.Nco(0.0, 0.1)
    for e in (-0.01, 0.02, 0.0, 6.0):
        assert abs(node.run(e) - orc.push(e)) <= 1e-15


# ------------------------------------------------------------------ C++ host mirror (graph-level conformance)
def test_cpp_host_graph_conformance():
    """comms-rs_b200/host/test_graph.cpp: source -> GPU node -> check graphs with one thread per
    node, expected values = the reference's golden vectors (the reference's own test pattern)."""
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    host = os.path.join(root, "comms-rs_b200", "host")
    subprocess.run(["make", "-C", host, "-s", "all"], check=True)
    r = subprocess.run([os.path.join(host, "test_graph")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "host graph tests ok" in r.stdout


# ------------------------------------------------------------------ bench.py --dump-outputs
def test_bench_dump_outputs_are_reproducible_and_are_what_the_path_computed(cb, oracle, tmp_path):
    """Two runs with the same arguments dump the same bytes, within the size limit, and the dumped rows of the headline
    FIR are its outputs at the positions bench.sample_rows names (last timed step: the state is the stream's tail)."""
    import importlib.util
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "3", "--no-e2e",
                            "--no-cpu", "--also", "freqest,fir64_iq16", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        files = sorted(os.listdir(d))
        assert files == ["fir64.npy", "fir64_iq16.npy", "freqest.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= bench.DUMP_BYTES
        dumps.append({f: np.load(d / f) for f in files})
    for f, a in dumps[0].items():
        assert a.dtype in (np.float32, np.float64) and a.tobytes() == dumps[1][f].tobytes(), f
    assert dumps[0]["freqest.npy"].shape == (1,) and dumps[0]["freqest.npy"].dtype == np.float64
    n = bench.WORKLOADS["fir64"][1]
    y = dumps[0]["fir64.npy"]
    assert y.shape[1] == 2 and 8 * len(y) <= bench.DUMP_BYTES // 3
    idx = bench.sample_rows(n, len(y))
    taps = bench.fir_taps("fir64")
    pick = [j for j in range(0, len(idx), len(idx) // 200) if idx[j] >= 63][:200]
    want = [oracle.batch_fir(oracle.synth_uniform_c32(bench.SEED, int(idx[j]) - 63, 64), taps, np.zeros(64, np.complex64))[0][-1]
            for j in pick]
    got = y[pick, 0] + 1j * y[pick, 1]
    assert rel_l2(got, want) <= FIR_TOL
