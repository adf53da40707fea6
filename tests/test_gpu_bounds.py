"""Every output of the FIR, chain and FM paths against a float64 per-output bound (tests/bounds.py).

The parity tests elsewhere use relative L2 (per frame or per 64-sample window) and, for FM, the median and the
fraction of large errors: a handful of wrong outputs passes them.  Here every output n must satisfy
|got_n - exact_n| <= 1e-5 * sum_k |h_k| |x_{n-k}| (FIR), or the FM angle bound derived from it, and the outputs
where the kernels differ from their steady state -- tile seams, call edges, the first tile's history -- are checked
on their own first so that a failure names them.  Needs a B200: `pytest -m gpu`.
"""
import zlib

import numpy as np
import pytest

import bounds as B

pytestmark = pytest.mark.gpu

TOL = 1e-5
TILE = 4096  # outputs per tile of the tensor-core FIR (fir_tc_kernel.cu)


@pytest.fixture(scope="module")
def cb():
    import comms_rs_b200 as m

    m.init(0)
    return m


def rnd_c32(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


def _lowpass(n):
    k = np.arange(n) - (n - 1) / 2
    return (np.sinc(k / 5) * np.hamming(n) / 5).astype(np.float32).astype(np.complex64)


def _taps(rng, ntaps, cplx, sparse, interp=1):
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    if sparse:  # every other tap (of every phase) zero: some outputs see only every other sample
        t[(np.arange(ntaps) // interp) % 2 == 1] = 0
    return t


def _seams(calls, tile):
    """first output of every call and of every tile inside it, and the output before each"""
    idx, s = [], 0
    for n in calls:
        for k in range(0, n, tile):
            idx += [s + k - 1, s + k]
        s += n
    return np.unique(np.clip(idx, 0, s - 1))


def _scale(x, lo, hi, e):
    x[lo:hi] *= np.float32(2.0 ** -e)


def _adversarial(rng, calls, tile=TILE):
    """loud / quiet interleaved samples, quiet stretches at 2^-16 .. 2^-30 inside a tile, across tile edges and across
    call boundaries, single tiny samples among loud ones, exact zeros (tiles of `tile` samples; the first call holds
    at least 14 of them)"""
    n = sum(calls)
    c1, c2 = calls[0], calls[0] + calls[1]
    x = rnd_c32(rng, n)
    x[1:tile:2] *= np.float32(2.0 ** -20)                 # interleaved, tile 0 (its history is zeros)
    x[tile + 1 : 3 * tile : 2] *= np.float32(2.0 ** -26)  # interleaved, tiles 1 and 2
    w = tile // 16
    for i, e in enumerate((16, 20, 24, 27, 30)):
        _scale(x, (3 + i) * tile + 6 * w, (3 + i) * tile + 10 * w, e)  # inside a tile
        _scale(x, (9 + i) * tile - w, (9 + i) * tile + w, e)            # across a tile edge
    _scale(x, c1 - 300, c1 + 300, 24)                                   # across the first call boundary
    _scale(x, c1 + 3 * tile - w, c1 + 3 * tile + w, 27)                 # across a tile edge of call 2
    _scale(x, c2 - 300, c2 + 300, 30)                                   # across the second call boundary
    for i, j in enumerate(range(c1 + 4 * tile, c2 - 2 * tile, 1009)):
        x[j] *= np.float32(2.0 ** -(20 + i % 11))                       # single tiny samples among loud ones
    x[c2 - 2 * tile + 100 : c2 - 2 * tile + 400] = 0                    # exact zeros are not quiet
    return x


def _run_calls(node_run, x, calls):
    out, s = [], 0
    for n in calls:
        out.append(node_run(x[s : s + n]))
        s += n
    return np.concatenate(out)


def _exact_calls(x, taps, calls, interp=1, decim=1, state=None):
    ys, As, s, st = [], [], 0, state
    for n in calls:
        y, st_next = B.fir64(x[s : s + n], taps, st, interp, decim)
        As.append(B.fir_mag64(x[s : s + n], taps, st, interp, decim))
        ys.append(y)
        st, s = st_next, s + n
    return np.concatenate(ys), np.concatenate(As), st


FIR_CALLS = (57_344, 45_057, 30_000)  # 14 whole tiles, then an odd call, then a short one


@pytest.mark.parametrize("path", ["tc", "cuda"])
@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("ntaps", [1, 2, 7, 32, 64, 100, 128])
def test_fir_every_output_within_bound(cb, ntaps, cplx, sparse, path, monkeypatch):
    # Tensor-core FIR (fp16 hi/lo split of a tile scaled by one power of two; tiles the split cannot carry are
    # recomputed in f32) and the CUDA-core direct form on the same adversarial stream, three calls.  With taps that
    # skip every other sample, outputs are formed from the quiet samples of an interleaved stretch alone: the quiet
    # test must look at single samples there, not at 16-byte pairs.
    monkeypatch.setenv("COMMS_B200_FIR_PATH", path)
    rng = np.random.default_rng(ntaps * 4 + cplx * 2 + sparse)
    taps = _taps(rng, ntaps, cplx, sparse)
    x = _adversarial(rng, FIR_CALLS)
    node = cb.BatchFirNode(taps)
    got = _run_calls(node.run, x, FIR_CALLS)
    exact, A, st = _exact_calls(x, taps, FIR_CALLS)
    what = f"{path} ntaps={ntaps} cplx={cplx} sparse={sparse}"
    B.assert_fir_bound(got, exact, A, TOL, what + " (tile seams / call edges)", idx=_seams(FIR_CALLS, TILE))
    B.assert_fir_bound(got, exact, A, TOL, what)
    assert node.state.tobytes() == st.astype(np.complex64).tobytes()


@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("L,ntaps,cplx", [(4, 32, False), (8, 1024, False), (8, 128, True), (4, 64, True)])
def test_polyphase_every_output_within_bound(cb, oracle, L, ntaps, cplx, sparse, monkeypatch):
    # polyphase bank on the tensor cores (fir_ptc_kernel.cu), f32 output and the fused i16 epilogue, same adversarial
    # stream at the symbol level
    monkeypatch.setenv("COMMS_B200_FIR_PATH", "tc")
    rng = np.random.default_rng(100 + L + ntaps + cplx + 7 * sparse)
    taps = _taps(rng, ntaps, cplx, sparse, L)
    calls = (15_360, 11_265, 7_500)
    sym = _adversarial(rng, calls, 1024)
    node = cb.BatchFirNode(taps, None, interp=L)
    got = _run_calls(node.run, sym, calls)
    exact, A, st = _exact_calls(sym, taps, calls, interp=L)
    what = f"ptc L={L} ntaps={ntaps} cplx={cplx} sparse={sparse}"
    B.assert_fir_bound(got, exact, A, TOL, what + " (call edges)", idx=_seams([c * L for c in calls], 1 << 40))
    B.assert_fir_bound(got, exact, A, TOL, what)
    assert node.state.tobytes() == st.astype(np.complex64).tobytes()
    scale = 1024.0
    twin = cb.BatchFirNode(taps, None, interp=L)
    i16 = _run_calls(lambda s: twin.run_i16(s, scale), sym, calls)
    assert np.array_equal(i16, oracle.quantize_i16(got, scale).reshape(-1, 2)), what + " (i16)"


def _state_with(kind, rng, nstate):
    st = rnd_c32(rng, nstate)
    if kind == "inf":
        st[5] = np.complex64(complex(np.inf, 0.25))
    elif kind == "nan":
        st[nstate // 2] = np.complex64(complex(0.5, np.nan))
    elif kind == "huge":  # 1e6 times the largest widened i16 sample
        st *= np.float32(1e6)
    elif kind == "denormal":
        st *= np.float32(1e-39)
    return st


@pytest.mark.parametrize("entry", ["host", "dev"])
@pytest.mark.parametrize("setup", ["set_state", "f32_call"])
@pytest.mark.parametrize("kind", ["inf", "nan", "huge", "denormal"])
def test_iq16_matches_three_step_after_any_history(cb, oracle, kind, setup, entry, monkeypatch):
    # cb_fir_run[_dev]_iq16 promises convert -> run -> quantize exactly.  Its fused kernel reads the first tile's halo
    # from the f32 history, which set_state or an f32 call can fill with anything: Inf / NaN, values far outside the
    # i16 range, denormals.  The words must equal the three-step form of a twin handle bit for bit, and so must the
    # carried state.  out_scale 2^14 with outputs ~0.2: an error of 1e-5 of an output moves it by ~0.03 LSB.
    import torch

    monkeypatch.setenv("COMMS_B200_FIR_PATH", "tc")
    rng = np.random.default_rng(zlib.crc32(f"{kind}/{setup}/{entry}".encode()))
    ntaps, n = 64, 50_000
    taps = (rnd_c32(rng, ntaps) / 16).astype(np.complex64)
    in_scale, out_scale = 1.0 / 32768, 16384.0
    iq = rng.integers(-32768, 32768, (n, 2), dtype=np.int16)
    a, b = cb.BatchFirNode(taps), cb.BatchFirNode(taps)
    if setup == "set_state":
        st = _state_with(kind, rng, ntaps)
        a.state = st
        b.state = st
    else:
        x0 = rnd_c32(rng, 1000)
        x0[-ntaps:] = _state_with(kind, rng, ntaps)[::-1]
        with np.errstate(all="ignore"):
            assert a.run(x0).tobytes() == b.run(x0).tobytes()
    if entry == "host":
        got = a.run_iq16(iq, in_scale, out_scale)
    else:
        d_in = torch.from_numpy(iq.reshape(-1).copy()).cuda()
        d_out = torch.empty(2 * n, dtype=torch.int16, device="cuda")
        torch.cuda.synchronize()
        assert a.run_dev_iq16(d_in.data_ptr(), n, in_scale, out_scale, d_out.data_ptr(), n) == n
        torch.cuda.synchronize()
        got = d_out.cpu().numpy().reshape(-1, 2)
    xf = (np.float32(in_scale) * iq.astype(np.float32)).view(np.complex64).reshape(-1)
    with np.errstate(all="ignore"):
        want = oracle.quantize_i16(b.run(xf), out_scale).reshape(-1, 2)
    diff = np.flatnonzero((got != want).any(axis=1))
    assert diff.size == 0, (f"{kind}/{setup}/{entry}: {diff.size} of {n} words differ from convert -> run -> quantize, "
                            f"first at {diff[:8].tolist()}")
    assert a.state.tobytes() == b.state.tobytes()


CHAIN_CALLS = (61_448, 40_024, 30_720)  # n_out 12290 / 8005 (odd: the next channel's row starts mid-word) / 6144 at D = 5


def _chain_exact(x, taps, D, dph, calls):
    """float64 mixer -> FIR -> per-call decimation of one channel over the calls, and the magnitudes A"""
    ys, As, s, st, ph = [], [], 0, None, 0.0
    for n in calls:
        xc = x[s : s + n]
        m, ph = B.mix64(xc, dph, ph) if dph is not None else (xc.astype(np.complex128), ph)
        y, st_next = B.fir64(m, taps, st, 1, D)
        As.append(B.fir_mag64(m, taps, st, 1, D))
        ys.append(y)
        st, s = st_next, s + n
    return np.concatenate(ys), np.concatenate(As)


@pytest.mark.parametrize("path,u8,mix,D", [("tc", True, False, 5), ("v3", True, False, 5), ("v3", True, True, 10),
                                          ("v3", False, True, 5), ("v3", False, False, 10), ("v3", True, True, 5)])
@pytest.mark.parametrize("fm", [True, False])
def test_chain_every_output_within_bound(cb, oracle, path, u8, mix, D, fm, monkeypatch):
    # fused mixer -> FIR -> decimate [-> FM] bank: chain_tc_kernel.cu (COMMS_B200_CHAIN_PATH=tc: bytes, D = 5, <= 64
    # real taps; the first discriminator output of every 2048-output tile comes from a separate seam kernel) and the
    # CUDA-core chain3 kernel (v3: tiles whose first output's predecessor is recomputed separately).  Three calls carry
    # the FIR history, the mixer phase and the FM predecessor; every FM output is held to the angle bound.  tc and v3 see
    # the same bytes (same seed) and each is checked against the float64 chain.
    monkeypatch.setenv("COMMS_B200_CHAIN_PATH", path)
    rng = np.random.default_rng(31 + D + 2 * mix + u8)
    C, taps = 3, _lowpass(63)
    dph = -2 * np.pi * rng.uniform(-0.4, 0.4, C) if mix else None
    bank = cb.ChainBank(C, taps, D, dphase=dph, with_fm=fm)
    outs, xs = [], []
    for n in CHAIN_CALLS:
        if u8:
            iq = rng.integers(0, 256, (C, n, 2), dtype=np.uint8)
            xs.append(oracle.u8_to_f32(iq.reshape(-1)).view(np.complex64).reshape(C, n))
            outs.append(bank.run_u8(iq))
        else:
            xs.append(rnd_c32(rng, C * n).reshape(C, n))
            outs.append(bank.run(xs[-1]))
    got, x = np.concatenate(outs, axis=1), np.concatenate(xs, axis=1)
    seams = _seams([-(-n // D) for n in CHAIN_CALLS], 128)  # 128 divides the tc kernel's 2048-output tiles
    for c in range(C):
        y, A = _chain_exact(x[c], taps, D, None if dph is None else dph[c], CHAIN_CALLS)
        what = f"chain {path} u8={u8} mix={mix} D={D} fm={fm} channel {c}"
        if fm:
            B.assert_fm_bound(got[c], y, A, TOL, what + " (tile seams / call edges)", idx=seams)
            B.assert_fm_bound(got[c], y, A, TOL, what)
        else:
            B.assert_fir_bound(got[c], y, A, TOL, what + " (tile seams / call edges)", idx=seams)
            B.assert_fir_bound(got[c], y, A, TOL, what)


SPLITS = (1, 2, 3, 5, 1, 4, 7, 1001, 2, 4099, 3, 40_000, 6, 1)  # prev_in at every position of the 4-wide loop


def test_fm_demod_node_every_output_within_bound(cb):
    # FMDemodNode (misc_kernels.cu): prev carried across calls of every length and alignment
    rng = np.random.default_rng(5)
    x = rnd_c32(rng, sum(SPLITS))
    node = cb.FMDemodNode()
    got = _run_calls(node.run, x, SPLITS)
    starts = np.cumsum((0,) + SPLITS[:-1])
    A = np.abs(x.astype(np.complex128))  # the input is exact: only the product and the angle round
    B.assert_fm_bound(got, x, A, 1e-6, "fm demod (call starts)", idx=starts)
    B.assert_fm_bound(got, x, A, 1e-6, "fm demod")


@pytest.mark.parametrize("D,ntaps", [(5, 63), (10, 63), (4, 17), (2, 64)])
def test_fir_real_decim_every_output_within_bound(cb, D, ntaps):
    # cb_fir_run_real: real in, real parts out, decimated per call, history carried across calls of every length
    rng = np.random.default_rng(D * 100 + ntaps)
    taps = _lowpass(ntaps)
    x = rng.uniform(-1, 1, sum(SPLITS)).astype(np.float32)
    x[20_000:20_500] *= np.float32(2.0 ** -24)
    node = cb.BatchFirNode(taps, None, decim=D)
    got = _run_calls(node.run_real, x, SPLITS)
    ys, As, s, st = [], [], 0, None
    for n in SPLITS:
        y, st_next = B.fir64(x[s : s + n], taps, st, 1, D)
        As.append(B.fir_mag64(x[s : s + n], taps, st, 1, D))
        ys.append(y.real)
        st, s = st_next, s + n
    outs = [-(-n // D) for n in SPLITS]
    B.assert_fir_bound(got, np.concatenate(ys), np.concatenate(As), TOL, f"fir_real D={D} (call starts)",
                       idx=np.cumsum([0] + outs[:-1]))
    B.assert_fir_bound(got, np.concatenate(ys), np.concatenate(As), TOL, f"fir_real D={D}")


def test_tap_dynamic_range_absolute_bound(cb, monkeypatch):
    # Documented exception (comms_b200.h): the tap image is split with ONE scale, so a tap far below the largest is
    # carried to ~2^-39 of the largest tap in absolute terms, not to 1e-5 of itself.  An isolated impulse through a tap
    # of 1e-8 of the maximum: the output is held to 2^-36 |h|max |x| absolute (8x the split's resolution).
    monkeypatch.setenv("COMMS_B200_FIR_PATH", "tc")
    taps = np.zeros(64, np.complex64)
    taps[0], taps[17] = 1.0, 1e-8
    x = np.zeros(20_000, np.complex64)
    x[5_000] = 1.0
    got = cb.BatchFirNode(taps).run(x).astype(np.complex128)
    exact, _ = B.fir64(x, taps)
    err = np.abs(got - exact)
    assert err.max() <= 2.0 ** -36, (int(np.argmax(err)), float(err.max()))
