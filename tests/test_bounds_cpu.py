"""The per-output bounds of tests/bounds.py, checked on the CPU: the f32 oracle meets them on adversarial inputs, they
reject single wrong outputs that the older metrics (relative L2 per 64-sample window, FM median and fraction) let
through, and an emulation of the tensor-core fp16 split shows why the quiet test must look at single samples for
parity-sparse taps."""
import numpy as np
import pytest

import bounds as B

TOL = 1e-5


def rnd_c32(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


def _lowpass(n):
    k = np.arange(n) - (n - 1) / 2
    return (np.sinc(k / 5) * np.hamming(n) / 5).astype(np.float32).astype(np.complex64)


def _input(kind, rng, n):
    x = rnd_c32(rng, n)
    if kind == "interleaved":  # loud / quiet alternating, quiet at 2^-17 .. 2^-30
        for i, e in enumerate(range(17, 31)):
            x[i * 1000 + 1 : (i + 1) * 1000 : 2] *= np.float32(2.0 ** -e)
    elif kind == "stretches":
        for i, e in enumerate(range(17, 31)):
            x[i * 1000 + 200 : i * 1000 + 700] *= np.float32(2.0 ** -e)
        x[15_000:15_300] = 0
    elif kind == "nonfinite":
        x[1234] = np.complex64(complex(np.inf, 0.5))
        x[7777] = np.complex64(complex(0.25, np.nan))
        x[9000] = np.complex64(complex(-np.inf, -np.inf))
    return x


# old metric of the FIR parity tests (tests/test_gpu_fuzz.py): relative L2 of every 64-sample window
def _windows_ok(got, want, win, tol):
    n = len(want) // win * win
    g = got[:n].astype(np.complex128).reshape(-1, win)
    w = want[:n].astype(np.complex128).reshape(-1, win)
    num = np.linalg.norm(g - w, axis=1)
    den = np.linalg.norm(w, axis=1)
    rel = np.where(den > 0, num / np.where(den > 0, den, 1), num)
    return bool(rel.max() <= tol)


# old metric of the FM parity tests (tests/test_gpu_parity.py, tests/test_gpu_fuzz.py)
def _fm_stats_ok(got, want):
    d = np.abs(got.astype(np.float64) - want.astype(np.float64))
    d = np.minimum(d, 2 * np.pi - d)
    return bool(np.median(d) < 2e-6 and np.mean(d > 1e-3) < 5e-3)


@pytest.mark.parametrize("kind", ["random", "interleaved", "stretches", "nonfinite"])
@pytest.mark.parametrize("interp,ntaps,cplx", [(1, 1, False), (1, 64, True), (1, 128, False), (4, 32, False), (8, 128, True)])
def test_oracle_fir_meets_bound(oracle, kind, interp, ntaps, cplx):
    rng = np.random.default_rng(ntaps + interp)
    taps = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    x = _input(kind, rng, 16_000)
    st32, st64 = np.zeros(ntaps, np.complex64), None
    for lo, hi in ((0, 5_001), (5_001, 5_003), (5_003, 16_000)):  # three calls, the state carried
        xu = oracle.upsample(x[lo:hi], interp) if interp > 1 else x[lo:hi]
        with np.errstate(all="ignore"):
            got, st32 = oracle.batch_fir(xu, taps, st32)
        exact, st64_next = B.fir64(x[lo:hi], taps, st64, interp)
        A = B.fir_mag64(x[lo:hi], taps, st64, interp)
        st64 = st64_next
        B.assert_fir_bound(got, exact, A, TOL, f"oracle {kind} calls [{lo}, {hi})")
    assert st32.tobytes() == st64.astype(np.complex64).tobytes()


@pytest.mark.parametrize("mix,D,u8", [(False, 5, True), (True, 10, True), (True, 5, False), (False, 10, False)])
def test_oracle_chain_meets_fm_bound(oracle, mix, D, u8):
    # fm_radio-style byte chain (ConvertNode -> 63-tap lowpass -> /D -> FM) and the mixer variants, three calls
    rng = np.random.default_rng(D + 2 * mix + u8)
    taps, dph = _lowpass(63), 0.7
    ref = oracle.FmChain(dph, 0.0, taps, D, do_mix=mix, do_fm=True)
    got, ys, As, st, ph = [], [], [], None, 0.0
    for n in (20_480, 10_243, 8_000):
        if u8:
            x = oracle.u8_to_f32(rng.integers(0, 256, 2 * n, dtype=np.uint8)).view(np.complex64)
        else:
            x = rnd_c32(rng, n)
        got.append(ref.run(x))
        m, ph = B.mix64(x, dph, ph) if mix else (x.astype(np.complex128), ph)
        y, st_next = B.fir64(m, taps, st, 1, D)
        As.append(B.fir_mag64(m, taps, st, 1, D))
        ys.append(y)
        st = st_next
    B.assert_fm_bound(np.concatenate(got), np.concatenate(ys), np.concatenate(As), TOL, "oracle chain")


def test_oracle_fm_demod_meets_bound(oracle):
    rng = np.random.default_rng(3)
    x = rnd_c32(rng, 50_000)
    fm = oracle.FM()
    got = np.concatenate([fm.demod(x[:1]), fm.demod(x[1:3]), fm.demod(x[3:30_001]), fm.demod(x[30_001:])])
    B.assert_fm_bound(got, x, np.abs(x.astype(np.complex128)), 1e-6, "oracle FM")


def test_fm_angle_fast_error_is_within_eps_atan():
    # EPS_ATAN is the measured error of fm_angle_fast (NumPy port) with margin; keep it honest
    rng = np.random.default_rng(11)
    s, p = rnd_c32(rng, 1 << 20), rnd_c32(rng, 1 << 20)
    r, tr, ti = B.fm_angle_fast_np(s, p)
    d = np.abs(r - np.arctan2(ti.astype(np.float64), tr.astype(np.float64)))
    d = np.minimum(d, 2 * np.pi - d)
    assert 1e-7 < d.max() <= B.EPS_ATAN


def test_one_quiet_fir_output_off_by_1e4_fails_bound_passes_windows(oracle):
    # a short quiet stretch (16 samples at 2^-20) through 4 taps: its quiet outputs share their 64-sample window with
    # loud ones
    rng = np.random.default_rng(21)
    taps = rnd_c32(rng, 4)
    x = rnd_c32(rng, 16_000)
    x[5_000:5_016] *= np.float32(2.0 ** -20)
    got, _ = oracle.batch_fir(x, taps, np.zeros(4, np.complex64))
    exact, _ = B.fir64(x, taps)
    A = B.fir_mag64(x, taps)
    B.assert_fir_bound(got, exact, A, TOL)
    j = 5_010
    bad = got.copy()
    bad[j] += np.complex64(1e-4 * abs(got[j]))
    assert _windows_ok(bad, got, 64, TOL)
    nbad, worst, ratio = B.fir_bound_report(bad, exact, A, TOL)
    assert nbad == 1 and worst == j and ratio > 2, (nbad, worst, ratio)


def _chain(oracle, calls, seed=4):
    rng = np.random.default_rng(seed)
    taps, D = _lowpass(63), 5
    ref = oracle.FmChain(0.0, 0.0, taps, D, do_mix=False, do_fm=True)
    xs = [oracle.u8_to_f32(rng.integers(0, 256, 2 * n, dtype=np.uint8)).view(np.complex64) for n in calls]
    got = [ref.run(x) for x in xs]
    ys, As, st = [], [], None
    for x in xs:
        y, st_next = B.fir64(x, taps, st, 1, D)
        As.append(B.fir_mag64(x, taps, st, 1, D))
        ys.append(y)
        st = st_next
    return xs, got, np.concatenate(ys), np.concatenate(As), taps, D


def test_one_fm_output_at_tile_seam_off_by_1e3_fails_bound_passes_stats(oracle):
    _, got, y, A, _, _ = _chain(oracle, (40_960,))
    got = got[0]
    B.assert_fm_bound(got, y, A, TOL)
    bad = got.copy()
    bad[2048] += np.float32(1e-3)  # the first output of the chain_tc kernel's second tile
    assert _fm_stats_ok(bad, got)
    nbad, worst, ratio, _ = B.fm_bound_report(bad, y, A, TOL)
    assert nbad == 1 and worst == 2048 and ratio > 1, (nbad, worst, ratio)


def test_second_call_from_zero_prev_fails_bound_passes_stats(oracle):
    xs, got, y, A, taps, D = _chain(oracle, (20_480, 20_480))
    B.assert_fm_bound(np.concatenate(got), y, A, TOL)
    # the same chain, but the FM predecessor of the second call lost (zero) instead of carried
    ref = oracle.FmChain(0.0, 0.0, taps, D, do_mix=False, do_fm=True)
    first = ref.run(xs[0])
    ref.prev[:] = 0
    bad = np.concatenate([first, ref.run(xs[1])])
    assert _fm_stats_ok(bad, np.concatenate(got))
    nbad, worst, ratio, _ = B.fm_bound_report(bad, y, A, TOL)
    assert nbad == 1 and worst == len(first), (nbad, worst, ratio)


# ---------------------------------------------------------------- fp16 split emulation of the tensor-core FIR
def _split(v, mx):
    """the kernels' exact power-of-two block scale (max into [2^14, 2^15)) and hi / lo fp16 split (subnormals kept)"""
    e = np.frexp(np.float32(mx))[1] - 1
    sc = np.float32(2.0 ** (14 - e))
    s = (v * sc).astype(np.float32)
    hi = s.astype(np.float16).astype(np.float32)
    lo = (s - hi).astype(np.float16).astype(np.float32)
    return hi.astype(np.float64), lo.astype(np.float64), float(sc)


def _emulate_tc_tile(x, taps):
    """one tile of fir_tc_kernel: Ahi*Bhi + Ahi*Blo + Alo*Bhi, per real component, unscaled (accumulated in f64)"""
    xr = np.concatenate([x.real, x.imag]).astype(np.float32)
    tr = np.concatenate([taps.real, taps.imag]).astype(np.float32)
    xh, xl, sx = _split(xr, np.abs(xr).max())
    th, tl, st = _split(tr, np.abs(tr).max())
    n, k = len(x), len(taps)
    Xh, Xl = xh[:n] + 1j * xh[n:], xl[:n] + 1j * xl[n:]
    Th, Tl = th[:k] + 1j * th[k:], tl[:k] + 1j * tl[k:]
    y = np.convolve(Xh, Th) + np.convolve(Xh, Tl) + np.convolve(Xl, Th)
    return y[:n] / (sx * st)


@pytest.mark.parametrize("quiet,min_ratio", [(1e-8, 2.0), (1e-10, 100.0)])
def test_pair_quiet_test_misses_parity_sparse_taps(quiet, min_ratio):
    # Loud and quiet samples alternate and every other tap is zero: the odd outputs are formed from quiet samples
    # alone.  The tile's quiet test over 16-byte pairs sees only loud pair maxima, so the tile is not sent to the
    # exact fall-back -- but the two-term split carries the quiet samples only to ~2^-39 of the tile maximum, far
    # outside 1e-5 of those outputs' own terms.  A per-sample test flags it; this is why filters with such taps
    # (FirTcPlan::sample_min) use it.
    rng = np.random.default_rng(8)
    taps = rng.uniform(-1, 1, 32).astype(np.complex64)
    taps[1::2] = 0
    assert B.parity_sparse(taps) and not B.parity_sparse(rng.uniform(-1, 1, 32))
    x = rnd_c32(rng, 4096)
    x[1::2] *= np.float32(quiet)
    pairs = np.maximum(np.abs(x.real), np.abs(x.imag)).reshape(-1, 2)
    mx = pairs.max()
    assert pairs.max(axis=1).min() >= mx * 2.0 ** -20  # the pair test does not flag the tile
    assert pairs.min() < mx * 2.0 ** -20                # the per-sample test does
    got = _emulate_tc_tile(x, taps)
    exact, _ = B.fir64(x, taps)
    A = B.fir_mag64(x, taps)
    nbad, worst, ratio = B.fir_bound_report(got, exact, A, TOL)
    assert nbad > 0 and worst % 2 == 1 and ratio > min_ratio, (nbad, worst, ratio)
    # dense taps on the same input: every output has a loud term, and the split is well inside the bound
    dense = rng.uniform(-1, 1, 32).astype(np.complex64)
    assert B.fir_bound_report(_emulate_tc_tile(x, dense), B.fir64(x, dense)[0], B.fir_mag64(x, dense), TOL)[0] == 0
