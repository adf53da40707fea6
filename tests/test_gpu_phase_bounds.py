"""Every output of the stand-alone mixer and of the NCO scan, and both f64 estimators, against the exact-phase bounds of
tests/bounds.py (stated in include/comms_b200.h).

The parity tests compare the mixer by relative L2 and the NCO with the oracle's own f64 recurrence at up to 2^20
samples; the estimators on short inputs and one pure tone.  Here:
- mixer: every output (windows of the 2^28-sample bench shape) within (C_MIX u32 + u64 (|phase0| + n dphase)) |x_n|,
  on the vector path (32-byte aligned) and the scalar path (8-byte offsets 1..3), past one grid-stride pass, with the
  phase carried over split calls and over the host path's chunks, and zero, subnormal, 2^+-60 and non-finite samples
  at quad and grid-stride seams;
- NCO: every output within the causal bound, into the second and third scan chunks, on the scalar (misaligned d_perr)
  path, over one-sample and mixed calls and set_phase; one NaN, +-Inf or 1e6 at thread, warp, tile and scan-chunk
  edges leaves every earlier output within the bound (and makes every later one, and the carried phase, NaN);
- estimators: random-phase and noise inputs, so that every term moves the estimate, at and past the 1184-block cap
  and the timing kernel's tile loop, spikes at the first and last sample and at every stride seam, 2^+-400 scaling.
Needs a B200: `pytest -m gpu`.
"""
import numpy as np
import pytest

import bounds as B

pytestmark = pytest.mark.gpu

TWO_PI = 2 * np.pi
MIX_PASS = 148 * 8 * 256 * 4  # samples of one grid-stride pass of the mixer's vector loop (1,212,416)
FREQ_CAP = 148 * 8 * 256 * 8  # the frequency estimator reaches its 1184 CTAs at n = 2,424,832
FREQ_STRIDE = 148 * 8 * 256
TIM_PASS = 148 * 8 * 1024  # the timing kernel's CTAs loop over tiles past n = 1,212,416


@pytest.fixture(scope="module")
def cb():
    import comms_rs_b200 as m

    m.init(0)
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t

    return t


def rnd_c64(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


# -------------------------------------------------------------------------------------------------------------- mixer
def mixer_stream(cb, torch, x, dphase, phase0, splits, path, offset=0):
    """run x through one MixerNode in calls of the given lengths; returns (outputs, carried-term list per sample)"""
    node = cb.MixerNode(dphase, phase0)
    d = node.dphase
    outs, carried, c, ph = [], [], 0.0, phase0
    pos = 0
    for m in splits:
        seg = x[pos: pos + m]
        if path == "run":
            y = node.run(seg)
        else:
            buf = torch.empty(2 * (m + 4), dtype=torch.float32, device="cuda")
            obuf = torch.empty(2 * (m + 4), dtype=torch.float32, device="cuda")
            buf[2 * offset: 2 * (offset + m)] = torch.from_numpy(seg.view(np.float32).copy()).cuda()
            torch.cuda.synchronize()  # run_dev without a stream runs on the node's own non-blocking stream
            node.run_dev(buf.data_ptr() + 8 * offset, m, obuf.data_ptr() + 8 * offset)
            torch.cuda.synchronize()
            y = obuf[2 * offset: 2 * (offset + m)].cpu().numpy().view(np.complex64)
        outs.append(y)
        carried.append(np.full(m, c))
        c += B.mix_carry(ph, m, d)
        ph = node.phase
        pos += m
    assert 0 <= node.phase < TWO_PI + 1e-9
    return np.concatenate(outs), np.concatenate(carried), d


def check_mixer(got, x, d, phase0, carried, what):
    """every output of a stream against the exact phase from its start; `carried`: the carried-phase term per sample"""
    n = np.arange(len(x))
    for c in np.unique(carried):  # one value per call
        idx = np.nonzero(carried == c)[0]
        fails, _, _ = _mix_report_at(got[idx], x[idx], d, phase0, n[idx], c)
        assert not fails, f"{what}: {fails[0]}"


def _mix_report_at(got, x, d, phase0, n, carried):
    """mix_bound_report for outputs at arbitrary stream indices n (windows): contiguous runs share one call"""
    n = np.asarray(n, np.int64)
    breaks = np.nonzero(np.diff(n) != 1)[0] + 1
    worst, fails = 0.0, []
    for a, b in zip(np.concatenate([[0], breaks]), np.concatenate([breaks, [len(n)]])):
        f, w, r = B.mix_bound_report(got[a:b], x[a:b], d, phase0, int(n[a]), carried)
        fails += f
        worst = max(worst, r)
    return fails, 0, worst


MIX_LENGTHS = list(range(1, 10)) + [4095, 4097, MIX_PASS + 15]


@pytest.mark.parametrize("path,offset", [("dev", 0), ("dev", 1), ("dev", 2), ("dev", 3), ("run", 0)])
@pytest.mark.parametrize("n", MIX_LENGTHS)
def test_mixer_lengths_and_paths(cb, torch, path, offset, n):
    rng = np.random.default_rng(n + offset)
    x = rnd_c64(rng, n)
    for dphase, phase0 in ((0.37, -3.0), (TWO_PI - 2.0 ** -20, 1e6)):
        got, car, d = mixer_stream(cb, torch, x, dphase, phase0, [n], path, offset)
        check_mixer(got, x, d, phase0, car, f"mixer {path}+{offset} n={n} d={dphase} p0={phase0}")


@pytest.mark.parametrize("dphase", [0.0, 2.0 ** -30, 0.37, np.pi, TWO_PI - 2.0 ** -20])
@pytest.mark.parametrize("phase0", [0.0, -3.0, 1e6])
def test_mixer_phase_grid_split_calls(cb, torch, dphase, phase0):
    n = MIX_PASS + 4099
    rng = np.random.default_rng(11)
    x = rnd_c64(rng, n)
    splits = [1, 2, 3, 4097, n - 4103]
    for path, off in (("dev", 0), ("dev", 1)):
        got, car, d = mixer_stream(cb, torch, x, dphase, phase0, splits, path, off)
        check_mixer(got, x, d, phase0, car, f"mixer {path}+{off} split d={dphase} p0={phase0}")


def test_mixer_run_longer_than_host_chunk(cb, torch):
    n = (1 << 22) + 4097  # the host path's chunk is 2^22 samples: the phase is carried between chunks
    rng = np.random.default_rng(12)
    x = rnd_c64(rng, n)
    got, car, d = mixer_stream(cb, torch, x, 0.37, 0.5, [n], "run")
    # advance_phase runs between the chunks too
    car = np.where(np.arange(n) >= 1 << 22, B.mix_carry(0.5, 1 << 22, d), 0.0)
    check_mixer(got, x, d, 0.5, car, "mixer run past one host chunk")


@pytest.mark.parametrize("offset", [0, 1])
def test_mixer_special_samples_at_seams(cb, torch, offset):
    n = MIX_PASS + 64
    rng = np.random.default_rng(13)
    x = rnd_c64(rng, n)
    seams = [0, 3, 4, 7, 1023, 1024, MIX_PASS - 1, MIX_PASS, MIX_PASS + 1, n - 1]
    vals = [0, np.float32(1e-42) * (1 + 1j), np.float32(2.0 ** 60) * (1 - 1j), np.float32(2.0 ** -60) * 1j,
            complex(np.inf, 0), complex(np.nan, 1), complex(1, -np.inf), 0, np.float32(1e-40), complex(0, np.nan)]
    for i, v in zip(seams, vals):
        x[i] = v
    x[MIX_PASS // 2: MIX_PASS // 2 + 4] = [np.float32(1e-45), 0, np.float32(2.0 ** 60), complex(np.nan, np.nan)]
    got, car, d = mixer_stream(cb, torch, x, TWO_PI - 2.0 ** -20, 1e6, [n], "dev", offset)
    check_mixer(got, x, d, 1e6, car, f"mixer special samples +{offset}")


def test_mixer_bench_shape_windows(cb, torch):
    """one call of 2^28 samples at dphase = 2 pi - 2^-20: windows at the start, at every grid-stride seam, and the
    last 2^20 samples, where u64 n dphase is largest (about 2 f32 ulps)"""
    n = 1 << 28
    g = torch.Generator(device="cuda").manual_seed(14)
    x = torch.rand(2 * n, device="cuda", generator=g, dtype=torch.float32) * 2 - 1
    y = torch.empty_like(x)
    node = cb.MixerNode(TWO_PI - 2.0 ** -20, 0.25)
    torch.cuda.synchronize()
    node.run_dev(x.data_ptr(), n, y.data_ptr())
    torch.cuda.synchronize()
    idx = [np.arange(0, 1 << 16), np.arange(n - (1 << 20), n)]
    for s in range(MIX_PASS, n - (1 << 20), MIX_PASS):
        idx.append(np.arange(s - 512, s + 512))
    idx = np.unique(np.concatenate(idx))
    ti = torch.from_numpy(idx).cuda()
    xs = torch.stack([x[2 * ti], x[2 * ti + 1]], 1).cpu().numpy().view(np.complex64).ravel()
    ys = torch.stack([y[2 * ti], y[2 * ti + 1]], 1).cpu().numpy().view(np.complex64).ravel()
    fails, _, worst = _mix_report_at(ys, xs, node.dphase, 0.25, idx, 0.0)
    assert not fails, f"mixer 2^28: {fails[0]}"
    del x, y


# ---------------------------------------------------------------------------------------------------------------- NCO
def dyadic_perr(rng, n):
    return rng.integers(-(1 << 30) + 1, 1 << 30, n) * 2.0 ** -40


class NcoStream:
    """exact reference of one NCO stream (phase_0, dphase) over calls: outputs k of the stream, S_k, calls_k"""

    def __init__(self, phase0, dphase):
        self.phase0, self.dphase = phase0, dphase
        self.perr = []

    def check(self, got, perr, call_starts, what, nonfinite_from=None):
        perr = np.asarray(perr, np.float64)
        n = len(perr)
        c, s = B.nco_exact(self.phase0, self.dphase, perr)
        S = np.cumsum(np.abs(np.where(np.isfinite(perr), perr, 0.0)))
        k = np.arange(n)
        calls = np.searchsorted(np.asarray(call_starts), k, side="right") - 1
        within = k - np.asarray(call_starts)[calls]
        bound = B.nco_bound(self.phase0, S, calls, within // B.NCO_CHUNK)
        fails, w, r = B.nco_bound_report(got, c, s, bound, nonfinite_from)
        assert not fails, f"{what}: " + "; ".join(fails)
        return r


def nco_dev(cb, torch, node, perr, misalign=False):
    n = len(perr)
    buf = torch.empty(n + 1, dtype=torch.float64, device="cuda")
    o = 1 if misalign else 0
    buf[o: o + n] = torch.from_numpy(np.ascontiguousarray(perr)).cuda()
    out = torch.empty(2 * n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    node.run_dev(buf.data_ptr() + 8 * o, n, out.data_ptr())
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.complex128)


NCO_LENGTHS = [1, 2047, 2048, 2049, (1 << 21) - 1, 1 << 21, (1 << 21) + 1, (1 << 22) + 3, 3 * (1 << 21) + 7]


@pytest.mark.parametrize("n", NCO_LENGTHS)
def test_nco_every_output_within_causal_bound(cb, torch, n):
    rng = np.random.default_rng(n)
    perr = dyadic_perr(rng, n)
    for path in ("dev", "misaligned", "run") if n <= (1 << 22) + 3 else ("dev", "misaligned"):
        dphase, phase0 = (TWO_PI - 2.0 ** -20, 1e6) if path != "run" else (0.123456789, -3.0)
        node = cb.NcoNode(dphase, phase0)
        st = NcoStream(phase0, node.dphase)
        got = node.run(perr) if path == "run" else nco_dev(cb, torch, node, perr, path == "misaligned")
        st.check(got, perr, [0], f"NCO {path} n={n}")
        # the carried phase is the exact phase after the last output, in [0, 2 pi)
        p = node.phase
        assert 0.0 <= p < TWO_PI, p
        c, s = B.nco_exact(phase0, node.dphase, perr[-1:], start=n - 1, prefix=tuple(
            a[-1:] for a in B.exact_prefix(perr)))
        e = B._err_ld(np.array([np.exp(1j * p)]), c, s)[0]
        assert e <= float(B.nco_bound(phase0, np.abs(perr).sum(), 1, (n - 1) // B.NCO_CHUNK)) + 2 * B.U64, (path, e)


def test_nco_one_sample_and_mixed_calls(cb, torch):
    rng = np.random.default_rng(21)
    sizes = [1] * 4096 + [2, 3, 2047, 2049, 7, 1 << 21, 5]
    n = sum(sizes)
    perr = dyadic_perr(rng, n)
    node = cb.NcoNode(0.37, 2.5)
    st = NcoStream(2.5, node.dphase)
    outs, starts, pos = [], [], 0
    for i, m in enumerate(sizes):
        starts.append(pos)
        seg = perr[pos: pos + m]
        outs.append(np.atleast_1d(node.run(seg[0]) if m == 1 and i % 2 else
                                  (node.run(seg) if i % 3 else nco_dev(cb, torch, node, seg))))
        pos += m
    st.check(np.concatenate(outs), perr, starts, "NCO 4096 one-sample calls, then mixed sizes")


def test_nco_set_phase_mid_stream(cb, torch):
    rng = np.random.default_rng(22)
    node = cb.NcoNode(0.37, 0.1)
    a, b = dyadic_perr(rng, 5000), dyadic_perr(rng, 70001)
    NcoStream(0.1, node.dphase).check(nco_dev(cb, torch, node, a), a, [0], "NCO before set_phase")
    node.phase = -2.0
    NcoStream(-2.0, node.dphase).check(nco_dev(cb, torch, node, b), b, [0], "NCO after set_phase")


# positions: first / middle / last sample of a thread's 8, of a warp, of a tile; and of a scan chunk
NCO_EDGE_N = 3 * 2048 + 17
NCO_EDGES = [0, 3, 7, 8 * 15 + 4, 255, 2048 + 1024, 2 * 2048 - 1, 2 * 2048, 3 * 2048 + 16]
NCO_CHUNK_N = (1 << 22) + 3
NCO_CHUNK_EDGES = [(1 << 21) - 1, 1 << 21, (1 << 21) + (1 << 20) + 3, (1 << 22) - 1]


@pytest.fixture(scope="module")
def nco_bases():
    """base dyadic perr and its exact reference for the two lengths (shared by every injected value)"""
    out = {}
    for n in (NCO_EDGE_N, NCO_CHUNK_N):
        perr = dyadic_perr(np.random.default_rng(23), n)
        pre = B.exact_prefix(perr)
        c, s = B.nco_exact(0.5, 0.37, perr, prefix=pre)
        out[n] = (perr, pre, c, s)
    return out


@pytest.mark.parametrize("value", [np.nan, np.inf, -np.inf, 1e6])
@pytest.mark.parametrize("n", [NCO_EDGE_N, NCO_CHUNK_N])
def test_nco_nonfinite_and_huge_perr_stay_causal(cb, torch, nco_bases, value, n):
    perr0, pre0, c0, s0 = nco_bases[n]
    for j in NCO_EDGES if n == NCO_EDGE_N else NCO_CHUNK_EDGES:
        perr = perr0.copy()
        perr[j] = value
        node = cb.NcoNode(0.37, 0.5)
        assert node.dphase == 0.37
        got = nco_dev(cb, torch, node, perr)
        S = np.cumsum(np.abs(perr))
        k = np.arange(n)
        bound = B.nco_bound(0.5, S, 0, k // B.NCO_CHUNK)
        if np.isfinite(value):
            ph, pl = B.dd_add(pre0[0][j:], pre0[1][j:], value, 0.0)  # the base prefix with perr0[j] -> value
            ph, pl = B.dd_add(ph, pl, -perr0[j], 0.0)
            c1, s1 = B.nco_exact(0.5, 0.37, perr[j:], start=j, prefix=(ph, pl))
            c, s = np.concatenate([c0[:j], c1]), np.concatenate([s0[:j], s1])
            fails, w, r = B.nco_bound_report(got, c, s, bound)
            assert 0.0 <= node.phase < TWO_PI
        else:
            fails, w, r = B.nco_bound_report(got, c0, s0, bound, nonfinite_from=j)
            assert np.isnan(node.phase), (j, node.phase)
        assert not fails, f"NCO perr[{j}] = {value}, n={n}: " + "; ".join(fails)


# --------------------------------------------------------------------------------------------- frequency estimator
def random_phase(rng, n, scale=1.0):
    return np.exp(2j * np.pi * rng.random(n)) * rng.uniform(0.5, 1.5, n) * scale


def check_freq(cb, torch, x, what, dev=True):
    S, T, (re, im) = B.freq_exact(x)
    E = B.C_FREQ * B.U64 * B.freq_depth(len(x)) * T
    ests = [("host", cb.frequency_offset_estimate(x))]
    if dev:
        d = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        torch.cuda.synchronize()
        ests.append(("dev", cb.frequency_offset_estimate_dev(d.data_ptr(), len(x))))
    worst = 0.0
    for p, est in ests:
        ok, r, skipped = B.est_bound_report(est, abs(S), E, B.angle_dd(re, im))
        assert ok, f"{what} ({p}): |est - arg S| / bound = {r:.3g}, est {est!r}, arg S {B.angle_dd(re, im)!r}"
        worst = max(worst, r)
    return worst


@pytest.mark.parametrize("n", [2, 3, 2047, 2049, FREQ_CAP - 1, FREQ_CAP + 1, (1 << 24) + 5, 3 * 303104 + 1])
def test_freq_random_phase(cb, torch, n):
    check_freq(cb, torch, random_phase(np.random.default_rng(n), n), f"freq random-phase n={n}")


@pytest.mark.parametrize("where", ["first", "last", "seams"])
def test_freq_spikes(cb, torch, where):
    n = FREQ_CAP + 5 * FREQ_STRIDE + 3
    x = random_phase(np.random.default_rng(31), n)
    pos = {"first": [0], "last": [n - 1], "seams": list(range(FREQ_STRIDE, n, FREQ_STRIDE))}[where]
    for i in pos:
        x[i] *= 2.0 ** 20  # enters the terms i - 1 and i, on either side of the seam
    check_freq(cb, torch, x, f"freq spike at {where}")


@pytest.mark.parametrize("e", [400, -400])
def test_freq_scaled(cb, torch, e):
    n = FREQ_CAP + 7
    check_freq(cb, torch, random_phase(np.random.default_rng(32), n, 2.0 ** e), f"freq scaled 2^{e}")


def test_freq_nan_and_alignment(cb, torch):
    x = random_phase(np.random.default_rng(33), 100000)
    x[77777] = complex(np.nan, 0)
    assert np.isnan(cb.frequency_offset_estimate(x))
    d = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    torch.cuda.synchronize()
    assert np.isnan(cb.frequency_offset_estimate_dev(d.data_ptr(), len(x)))
    # d_samples is read as double2: an 8-byte offset is rejected before any launch
    with pytest.raises(cb.CbError):
        cb.frequency_offset_estimate_dev(d.data_ptr() + 8, len(x) - 1)


# ----------------------------------------------------------------------------------------------- timing estimator
def qpsk(rng, n, N):
    s = (rng.choice([-1.0, 1.0], -(-n // N)) + 1j * rng.choice([-1.0, 1.0], -(-n // N))) / np.sqrt(2)
    return np.repeat(s, N)[:n] + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))


TIMING_CASES = [(10, 5, "noise"), (10, 5, "qpsk"), (8, 0, "noise"), (3, 2, "noise"), (8, 256, "noise")]


@pytest.mark.parametrize("N,D,kind", TIMING_CASES)
def test_timing_every_length(cb, torch, N, D, kind):
    rng = np.random.default_rng(N * 1000 + D)
    ntaps = 2 * N * D + 1
    nd = N * D
    lengths = [nd, nd + 1, 1023, 1025, TIM_PASS - 1, TIM_PASS + 1]
    if ntaps <= 101:
        lengths.append(2_500_000)
    nmax = max(lengths)
    x = qpsk(rng, nmax, N) if kind == "qpsk" else (rng.standard_normal(nmax) + 1j * rng.standard_normal(nmax))
    taps = B.timing_taps(N, D, 0.5)
    S, W = B.timing_exact(x, taps, N, D)
    est = cb.TimingEstimator(N, D, 0.5)
    dx = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    torch.cuda.synchronize()  # push_dev without a stream runs on the estimator's own non-blocking stream
    scale = -N / (2 * np.pi)
    for n in lengths:
        if n == 0 or n <= nd:
            Sn, Wn = 0j, 0.0
        else:
            Sn, Wn = complex(S[n - 1]), float(W[n - 1])
        E = B.timing_E(n, ntaps, Wn)
        for p, got in (("host", est.push(x[:n])), ("dev", est.push_dev(dx.data_ptr(), n))):
            ok, r, skipped = B.est_bound_report(got, abs(Sn), E, float(np.angle(Sn)), scale)
            assert ok, f"timing N={N} D={D} {kind} n={n} ({p}): ratio {r:.3g}, est {got!r}"
    with pytest.raises(cb.CbError):
        est.push_dev(dx.data_ptr() + 8, 1000)
