"""Every output of the Complex<f64> FIR (cb_fir_f64, BatchFirNodeF64 / PulseNodeF64) against the CPU emulation of its
operation order (tests/emul/fir_f64_emul.cpp): bit for bit, NaN positions compared as NaN, non-finite exactly where an
output's taps reach a non-finite sample, and within the bound |y_n - y_exact| <= 3 K_n u A_n + K_n 2^-1072 of the
__float128 reference (include/comms_b200.h).

The seams named below are the kernels' own: the stream kernel's tiles of TILE outputs and chunks of TAP_CHUNK taps,
its grid-stride pass of STREAM_PASS outputs, and the resampling kernel's pass of RESAMPLE_PASS outputs.
Needs a B200: `pytest -m gpu`.
"""
import numpy as np
import pytest

import fir64_bounds as B

pytestmark = pytest.mark.gpu

TILE = 256 * 8                   # stream kernel: 256 threads x 8 consecutive outputs
TAP_CHUNK = 1024                 # taps staged per shared-memory chunk
STREAM_PASS = 148 * 4 * TILE     # 1,212,416 outputs: the stream kernel's CTAs loop over tiles past this
RESAMPLE_PASS = 148 * 16 * 256   # 606,208 outputs: one grid-stride pass of the resampling kernel

TAP_COUNTS = [1, 2, 3, 63, 64, 65, 101, 127, 128, 129, 1024, 1025, 4097]
RATIOS = {}  # shape -> worst err / bound seen


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
    return B.fir64_emul_lib(tmp_path_factory.mktemp("fir64_emul"))


def rnd(rng, n, scale=1.0):
    return scale * (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n))


def taps_of(rng, k, real):
    t = rng.standard_normal(k) * np.exp(-np.linspace(0, 3, k))
    return t.astype(np.complex128) if real else t + 1j * rng.standard_normal(k) * np.exp(-np.linspace(0, 3, k))


def to_dev(torch, x, pad=0):
    """complex128 host array -> float64 device tensor (2 (len + pad) doubles); returns (tensor, base pointer)"""
    t = torch.zeros(2 * (len(x) + pad), dtype=torch.float64, device="cuda")
    if len(x):
        t[: 2 * len(x)] = torch.from_numpy(np.ascontiguousarray(x).view(np.float64)).cuda()
    return t


def run_dev(torch, node, x, calls=None, stream=0):
    calls = [len(x)] if calls is None else calls
    outs, pos = [], 0
    for m in calls:
        xi = to_dev(torch, x[pos: pos + m])
        cap = node.out_len(m)
        yo = torch.empty(2 * max(cap, 1), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()  # run_dev without a stream runs on the node's own non-blocking stream
        n = node.run_dev(xi.data_ptr(), m, yo.data_ptr(), cap, stream)
        torch.cuda.synchronize()
        assert n == cap
        outs.append(yo[: 2 * n].cpu().numpy().view(np.complex128))
        pos += m
    return np.concatenate(outs) if outs else np.zeros(0, np.complex128)


def run_host(node, x, calls=None):
    calls = [len(x)] if calls is None else calls
    outs, pos = [], 0
    for m in calls:
        outs.append(node.run(x[pos: pos + m]))
        pos += m
    return np.concatenate(outs)


def check(got, emu, what, shape=None):
    B.fir64_check(got, emu, what)
    if emu.err is not None and shape is not None:
        RATIOS[shape] = max(RATIOS.get(shape, 0.0), emu.ratio())


# ----------------------------------------------------------------------------------------------- tap counts, lengths
@pytest.mark.parametrize("real", [True, False], ids=["real", "cplx"])
@pytest.mark.parametrize("k", TAP_COUNTS)
def test_tap_counts(cb, torch, emul, k, real):
    rng = np.random.default_rng(k)
    t = taps_of(rng, k, real)
    x = rnd(rng, 3 * TILE + 17)
    node = cb.BatchFirNodeF64(t)
    got = run_dev(torch, node, x)
    check(got, B.Fir64Emul(emul, t, x), f"{k} taps {'real' if real else 'complex'}", f"plain K={k} {'real' if real else 'cplx'}")


@pytest.mark.parametrize("real", [True, False], ids=["real", "cplx"])
@pytest.mark.parametrize("n", list(range(1, 10)) + [TILE - 1, TILE, TILE + 1])
def test_lengths(cb, torch, emul, n, real):
    rng = np.random.default_rng(n)
    t = taps_of(rng, 64, real)
    x = rnd(rng, n)
    got = run_dev(torch, cb.BatchFirNodeF64(t), x)
    check(got, B.Fir64Emul(emul, t, x), f"n={n}", f"plain K=64 {'real' if real else 'cplx'}")


@pytest.mark.parametrize("real", [True, False], ids=["real", "cplx"])
def test_past_one_grid_stride_pass(cb, torch, emul, real):
    rng = np.random.default_rng(5)
    t = taps_of(rng, 65, real)
    n = 2 * STREAM_PASS + 3 * TILE + 5
    x = rnd(rng, n)
    got = run_dev(torch, cb.BatchFirNodeF64(t), x)
    check(got, B.Fir64Emul(emul, t, x, exact=False), "bits past the grid-stride pass")
    for s in (STREAM_PASS, 2 * STREAM_PASS, n - 2 * TILE):  # the bound on windows around each pass seam
        lo = s - TILE
        emu = B.Fir64Emul(emul, t, x[lo: s + TILE], state=x[lo - 65: lo][::-1])
        check(got[lo: s + TILE], emu, f"window at {s}", f"plain K=65 {'real' if real else 'cplx'}")


# ------------------------------------------------------------------------------------------------------ split calls
@pytest.mark.parametrize("k,real", [(64, True), (65, False), (1025, False)])
def test_split_calls_and_host_entry(cb, torch, emul, k, real):
    rng = np.random.default_rng(k + 7)
    t = taps_of(rng, k, real)
    calls = [1, 2, 3, 1, 7, 1001, TILE - 1, 3, TILE + 1, 5, 2 * TILE + 3, 9]
    x = rnd(rng, sum(calls))
    emu = B.Fir64Emul(emul, t, x, calls=calls)
    one = run_dev(torch, cb.BatchFirNodeF64(t), x)
    check(one, emu, "one call", f"plain K={k} {'real' if real else 'cplx'}")
    check(run_dev(torch, cb.BatchFirNodeF64(t), x, calls), emu, "split device calls")
    check(run_host(cb.BatchFirNodeF64(t), x, calls), emu, "split host calls")
    check(run_host(cb.BatchFirNodeF64(t), x), emu, "one host call")
    f = cb.FirNodeF64(t)
    ys = np.array([f.run(v) for v in x[:40]])
    check(ys, B.Fir64Emul(emul, t, x[:40]), "FirNodeF64 one sample per run")


@pytest.mark.parametrize("D,L", [(1, 1), (3, 1), (1, 4)])
def test_host_chunks(emul, tmp_path, D, L):
    # the host entry pipelines chunks of 2^COMMS_B200_HOST_CHUNK_LOG2 samples, each re-sent with its predecessor's tail
    # as history; at 4096-sample chunks a 3-chunk call must give the same bits as the emulation of one call
    import os
    import subprocess
    import sys

    rng = np.random.default_rng(D * 10 + L)
    t = taps_of(rng, 65, False)
    x = rnd(rng, 3 * 4096 + 5)
    np.save(tmp_path / "t.npy", t)
    np.save(tmp_path / "x.npy", x)
    code = ("import sys, numpy as np, comms_rs_b200 as cb\n"
            "cb.init(0)\n"
            "d = sys.argv[1]\n"
            f"node = cb.BatchFirNodeF64(np.load(d + '/t.npy'), decim={D}, interp={L})\n"
            "np.save(d + '/y.npy', node.run(np.load(d + '/x.npy')))\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, COMMS_B200_HOST_CHUNK_LOG2="12", PYTHONPATH=root)
    subprocess.run([sys.executable, "-c", code, str(tmp_path)], env=env, check=True, cwd=root)
    check(np.load(tmp_path / "y.npy"), B.Fir64Emul(emul, t, x, decim=D, interp=L), f"host chunks D={D} L={L}")


# ------------------------------------------------------------------------------------------------------- decimation
@pytest.mark.parametrize("D", [2, 3, 5, 8, 10, 17])
@pytest.mark.parametrize("k,real", [(63, True), (64, False)])
def test_decimation(cb, torch, emul, D, k, real):
    rng = np.random.default_rng(D * 100 + k)
    t = taps_of(rng, k, real)
    calls = [4097, 1000, 3, 2 * TILE + 1]
    x = rnd(rng, sum(calls))
    emu = B.Fir64Emul(emul, t, x, calls=calls, decim=D)
    got = run_dev(torch, cb.BatchFirNodeF64(t, decim=D), x, calls)
    check(got, emu, f"decim {D}", f"decim {D} K={k} {'real' if real else 'cplx'}")
    check(run_host(cb.BatchFirNodeF64(t, decim=D), x, calls), emu, f"decim {D} host")
    plain = run_dev(torch, cb.BatchFirNodeF64(t), x, calls)
    pos, want = 0, []
    for m in calls:  # the decimation phase restarts at every call
        want.append(plain[pos: pos + m][::D])
        pos += m
    want = np.concatenate(want)
    assert got.view(np.uint64).tobytes() == want.view(np.uint64).tobytes(), "decimated != every D-th plain output"


def test_decimation_past_one_grid_stride_pass(cb, torch, emul):
    rng = np.random.default_rng(17)
    t = taps_of(rng, 63, True)
    n = 2 * RESAMPLE_PASS + 1001
    x = rnd(rng, n)
    got = run_dev(torch, cb.BatchFirNodeF64(t, decim=2), x)
    check(got, B.Fir64Emul(emul, t, x, decim=2, exact=False), "decim 2 past the resampling pass")


# ---------------------------------------------------------------------------------------------------- interpolation
@pytest.mark.parametrize("L", [2, 3, 4, 8])
@pytest.mark.parametrize("k,real", [(33, False), (64, True)])
def test_interpolation(cb, torch, emul, L, k, real):
    rng = np.random.default_rng(L * 10 + k)
    t = taps_of(rng, k, real)
    calls = [1, 2, 501, 3, 1000]
    x = rnd(rng, sum(calls))
    emu = B.Fir64Emul(emul, t, x, calls=calls, interp=L)
    check(run_dev(torch, cb.BatchFirNodeF64(t, interp=L), x, calls), emu, f"interp {L}", f"interp {L} K={k} {'real' if real else 'cplx'}")
    check(run_host(cb.BatchFirNodeF64(t, interp=L), x, calls), emu, f"interp {L} host")


@pytest.mark.parametrize("L,D", [(3, 2), (8, 5), (2, 3)])
def test_interp_and_decim(cb, torch, emul, L, D):
    rng = np.random.default_rng(L * 7 + D)
    t = taps_of(rng, 47, False)
    calls = [1, 7, 999, 2]
    x = rnd(rng, sum(calls))
    emu = B.Fir64Emul(emul, t, x, calls=calls, interp=L, decim=D)
    check(run_dev(torch, cb.BatchFirNodeF64(t, decim=D, interp=L), x, calls), emu, f"L={L} D={D}", f"L={L} D={D} K=47 cplx")


def test_pulse_node_rrc_1024_x8(cb, torch, emul):
    t = cb.rrc_taps(1024, 8, 0.25, dtype=np.complex128)
    rng = np.random.default_rng(8)
    sym = (2.0 * rng.integers(0, 2, 600) - 1).astype(np.complex128)
    p = cb.PulseNodeF64(t, 8)
    one_by_one = np.concatenate([p.run(s) for s in sym[:40]])
    rest = p.run(sym[40:])
    emu = B.Fir64Emul(emul, t, sym, calls=[1] * 40 + [560], interp=8)
    check(np.concatenate([one_by_one, rest]), emu, "PulseNodeF64", "interp 8 K=1024 real (rrc)")
    d = cb.PulseNodeF64(t, 8)
    check(run_dev(torch, d, sym), emu, "PulseNodeF64 run_dev")


# ------------------------------------------------------------------------------------------------------------ state
@pytest.mark.parametrize("nstate", [None, 64, 20, 150])
def test_state(cb, torch, emul, nstate):
    rng = np.random.default_rng(3 if nstate is None else nstate)
    t = taps_of(rng, 64, False)
    st = None if nstate is None else rnd(rng, nstate)
    calls = [100, TILE + 3]
    x = rnd(rng, sum(calls))
    node = cb.BatchFirNodeF64(t, state=st)
    got = run_dev(torch, node, x, calls)
    check(got, B.Fir64Emul(emul, t, x, calls=calls, state=st), f"nstate={nstate}", "plain K=64 cplx")
    # the carried state is the last nstate samples of [state ++ x], newest first (zeros of len taps for None)
    ns = 64 if nstate is None else nstate
    full = np.concatenate([np.zeros(ns, np.complex128) if st is None else st[::-1], x])
    want = full[::-1][:ns]
    assert node.state.tobytes() == want.tobytes()
    # round trip: set a state, run, compare with a fresh handle created with that state
    s2 = rnd(rng, ns)
    node.state = s2
    assert node.state.tobytes() == s2.tobytes()
    y2 = run_dev(torch, node, x[:500])
    check(y2, B.Fir64Emul(emul, t, x[:500], state=s2), "after set_state")


def test_interp_state_on_grid_and_off_grid(cb, torch, emul):
    rng = np.random.default_rng(11)
    t = taps_of(rng, 32, True)
    st = np.zeros(32, np.complex128)
    st[3::4] = rnd(rng, 8)  # on the symbol grid of L = 4
    x = rnd(rng, 300)
    node = cb.BatchFirNodeF64(t, state=st, interp=4)
    check(run_dev(torch, node, x), B.Fir64Emul(emul, t, x, state=st, interp=4), "interp state on grid")
    stuffed = np.concatenate([st[::-1], np.ravel(np.column_stack([x] + [np.zeros_like(x)] * 3))])
    assert node.state.tobytes() == stuffed[::-1][:32].tobytes()
    bad = st.copy()
    bad[0] = 1.0
    with pytest.raises(cb.CbError) as e:
        cb.BatchFirNodeF64(t, state=bad, interp=4)
    assert e.value.status == cb._lib.CB_ERR_UNSUPPORTED
    with pytest.raises(cb.CbError) as e:
        node.state = bad
    assert e.value.status == cb._lib.CB_ERR_UNSUPPORTED


@pytest.mark.parametrize("k,real", [(64, True), (1025, False)])
def test_segments_seeded_with_the_previous_tail(cb, torch, emul, k, real):
    # what sharding.py relies on: a second handle seeded with the first segment's tail continues the stream exactly
    rng = np.random.default_rng(k)
    t = taps_of(rng, k, real)
    x = rnd(rng, 3 * TILE + 11)
    s = TILE + 77
    one = run_dev(torch, cb.BatchFirNodeF64(t), x)
    a = run_dev(torch, cb.BatchFirNodeF64(t), x[:s])
    b = run_dev(torch, cb.BatchFirNodeF64(t, state=x[:s][::-1][:k]), x[s:])
    assert np.concatenate([a, b]).view(np.uint64).tobytes() == one.view(np.uint64).tobytes()
    check(one, B.Fir64Emul(emul, t, x), "one handle")


# ---------------------------------------------------------------------------------------------------- special values
@pytest.mark.parametrize("real", [True, False], ids=["real", "cplx"])
def test_zeros_subnormals_and_scaling(cb, torch, emul, real):
    rng = np.random.default_rng(21)
    t = taps_of(rng, 65, real)
    z = np.zeros(TILE + 5, np.complex128)
    got = run_dev(torch, cb.BatchFirNodeF64(t), z)
    assert (got.view(np.float64) == 0).all()
    for scale, name in ((2.0 ** -1060, "subnormal"), (2.0 ** 500, "2^500"), (2.0 ** -500, "2^-500")):
        x = rnd(rng, TILE + 5, scale)
        got = run_dev(torch, cb.BatchFirNodeF64(t), x)
        check(got, B.Fir64Emul(emul, t, x), name, f"{name} K=65 {'real' if real else 'cplx'}")
    x = rnd(rng, TILE + 5)
    x[100:400] = 0.0  # a silent stretch: outputs fully inside it are exactly 0
    x[1000:1200] *= 2.0 ** -1070
    got = run_dev(torch, cb.BatchFirNodeF64(t), x)
    check(got, B.Fir64Emul(emul, t, x), "silent and subnormal stretches")


@pytest.mark.parametrize("bad", [np.inf, -np.inf, np.nan, complex(0, np.inf), complex(np.nan, 0)], ids=str)
@pytest.mark.parametrize("k,real", [(63, True), (64, False), (1025, False)])
def test_non_finite_samples(cb, torch, emul, bad, k, real):
    rng = np.random.default_rng(31)
    t = taps_of(rng, k, real)
    calls = [TILE + 700, 3 * TILE]
    x = rnd(rng, sum(calls))
    # a tile seam, the call edge, and a sample whose reach ends exactly one output before the next seam
    for p in (TILE, calls[0], calls[0] + 2 * TILE - k):
        x[p] = bad
    emu = B.Fir64Emul(emul, t, x, calls=calls)
    assert emu.bad.sum() == 3 * k or k > 700
    check(run_dev(torch, cb.BatchFirNodeF64(t), x, calls), emu, f"non-finite {bad}")
    check(run_host(cb.BatchFirNodeF64(t), x, calls), emu, f"non-finite {bad} host")
    for D, L in ((5, 1), (1, 4)):
        e2 = B.Fir64Emul(emul, t, x, calls=calls, decim=D, interp=L)
        check(run_dev(torch, cb.BatchFirNodeF64(t, decim=D, interp=L), x, calls), e2, f"non-finite {bad} D={D} L={L}")


# -------------------------------------------------------------------------------------------------- errors, streams
def test_errors(cb, torch):
    t = taps_of(np.random.default_rng(1), 16, False)
    node = cb.BatchFirNodeF64(t)
    n = 100
    xi = torch.zeros(2 * (n + 2), dtype=torch.float64, device="cuda")
    yo = torch.zeros(2 * (n + 2), dtype=torch.float64, device="cuda")
    for dx, dy in ((8, 0), (0, 8), (8, 8)):
        with pytest.raises(cb.CbError) as e:
            node.run_dev(xi.data_ptr() + dx, n, yo.data_ptr() + dy, n)
        assert e.value.status == cb._lib.CB_ERR_INVALID_ARG and "aligned" in str(e.value)
    with pytest.raises(cb.CbError) as e:
        node.run_dev(xi.data_ptr(), n, xi.data_ptr() + 16, n)
    assert e.value.status == cb._lib.CB_ERR_INVALID_ARG and "overlap" in str(e.value)
    with pytest.raises(cb.CbError) as e:
        node.run_dev(xi.data_ptr(), n, yo.data_ptr(), n - 1)
    assert e.value.status == cb._lib.CB_ERR_SIZE
    for v in (np.inf, -np.inf, np.nan, complex(1, np.nan), complex(0, -np.inf)):
        tt = t.copy()
        tt[7] = v
        with pytest.raises(cb.CbError) as e:
            cb.BatchFirNodeF64(tt)
        assert e.value.status == cb._lib.CB_ERR_INVALID_ARG
    with pytest.raises(cb.CbError) as e:
        cb.BatchFirNodeF64(t, state=np.ones(10, np.complex128)).state = np.ones(9, np.complex128)
    assert e.value.status == cb._lib.CB_ERR_SIZE


def test_calls_on_two_streams_are_ordered_like_one(cb, torch, emul):
    rng = np.random.default_rng(41)
    t = taps_of(rng, 129, False)
    calls = [STREAM_PASS // 2 + 3, 4 * TILE + 1, 77]
    x = rnd(rng, sum(calls))
    node = cb.BatchFirNodeF64(t)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    xs, ys, pos = [], [], 0
    for m in calls:
        xs.append(to_dev(torch, x[pos: pos + m]))
        ys.append(torch.empty(2 * m, dtype=torch.float64, device="cuda"))
        pos += m
    torch.cuda.synchronize()
    for i, m in enumerate(calls):  # alternate streams, no host synchronisation between the calls
        node.run_dev(xs[i].data_ptr(), m, ys[i].data_ptr(), m, (s1 if i % 2 == 0 else s2).cuda_stream)
    torch.cuda.synchronize()
    got = np.concatenate([y.cpu().numpy().view(np.complex128) for y in ys])
    check(got, B.Fir64Emul(emul, t, x, calls=calls, exact=False), "two streams")


# ------------------------------------------------------------------------------------------------------- large call
def test_one_call_of_2_30_plus_5_samples(cb, torch, emul):
    n = (1 << 30) + 5
    k = 64
    rng = np.random.default_rng(51)
    t = taps_of(rng, k, False)
    g = torch.Generator(device="cuda").manual_seed(5)
    xd = torch.rand(2 * n, dtype=torch.float64, device="cuda", generator=g).mul_(2).sub_(1)  # 16 GiB in
    yd = torch.empty(2 * n, dtype=torch.float64, device="cuda")                       # 16 GiB out
    node = cb.BatchFirNodeF64(t)
    torch.cuda.synchronize()
    assert node.run_dev(xd.data_ptr(), n, yd.data_ptr(), n) == n
    torch.cuda.synchronize()
    last_tile = (n - 1) // TILE * TILE
    for lo, hi in ((0, 2 * TILE), ((1 << 30) - 3 * TILE, (1 << 30) + 5), ((1 << 31) // 2 - 7, (1 << 30) + 3),
                   (last_tile - TILE, n)):
        s0 = max(lo - k, 0)
        xw = xd[2 * s0: 2 * hi].cpu().numpy().view(np.complex128)
        st = xw[: lo - s0][::-1] if lo > 0 else None
        emu = B.Fir64Emul(emul, t, xw[lo - s0:], state=st)
        check(yd[2 * lo: 2 * hi].cpu().numpy().view(np.complex128), emu, f"window [{lo}, {hi})", "plain K=64 cplx")
    st = node.state
    assert st.tobytes() == xd[2 * (n - k): 2 * n].cpu().numpy().view(np.complex128)[::-1].tobytes()
    del xd, yd
    torch.cuda.empty_cache()


def test_report_worst_ratios():
    # the worst err / bound per shape seen by the tests above (run with -s to see it)
    for shape, r in sorted(RATIOS.items()):
        print(f"fir_f64 worst bound ratio  {shape:40s} {r:.3e}")
        assert r <= 1.0
