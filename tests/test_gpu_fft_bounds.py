"""Every bin of every frame of every FFT plan, and every output of the overlap-save FIR, against the float64 bounds of
tests/bounds.py.

The parity tests check relative L2 <= 1e-4 per frame, often on a few sampled frames with the rest checked by Parseval:
one wrong bin, one wrong intermediate of a two-step split or bins at the wrong indices pass them.  Here every bin must
satisfy |got_k - X_k| <= tau S_f (+ a floor for subnormal frames), every frame ||got - X|| <= rho ||X||, zero frames
give exact zeros and a non-finite input stays inside its own frame.  Inputs: impulses (every position up to 4096
points, digit and tile edges above), tones on exact bins, random frames, and batches that put zero, subnormal,
2^+-60-scaled, Inf and NaN frames next to each other at the CTA, cluster, ring-slot and chirp-z group boundaries.
Switches that the library reads once per process run in a child interpreter.  Needs a B200: `pytest -m gpu`.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import bounds as B

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNK = 1 << 22  # points per float64 check (the reference of one call stays near 256 MB)


@pytest.fixture(scope="module")
def cb():
    import comms_rs_b200 as m

    m.init(0)
    return m


def rnd_c32(rng, n):
    return (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)


def check(got, x, n, inverse, what, path=None):
    """every bin of every frame, in chunks of whole frames; prints the worst ratios (<= 1 passes)"""
    path = path or B.fft_path(n)
    per = max(1, CHUNK // n)
    x, got = np.asarray(x).reshape(-1, n), np.asarray(got).reshape(-1, n)
    wb = wn = 0.0
    for f0 in range(0, x.shape[0], per):
        fails, b, m = B.fft_bound_report(got[f0:f0 + per], x[f0:f0 + per], n, inverse, path)
        fails = [s.replace("frame ", f"frame {f0}+", 1) for s in fails]
        assert not fails, f"{what}: {len(fails)} failures; " + "; ".join(fails[:6])
        wb, wn = max(wb, b), max(wn, m)
    print(f"RATIO {what} {path} N={n} inv={int(inverse)} bin={wb:.3f} norm={wn:.3f}")


def impulses(n, positions):
    x = np.zeros((len(positions), n), np.complex64)
    x[np.arange(len(positions)), positions] = 1
    return x.ravel()


def impulse_positions(n, rng, n1=None):
    """every position up to 4096 points; above, digit and tile edges (16, 256, the split's N1) and random ones"""
    if n <= 4096:
        return np.arange(n)
    p = {0, 1, 15, 16, 17, 255, 256, 257, 4095, 4096, n // 2 - 1, n // 2, n // 2 + 1, n - 16, n - 1}
    if n1:
        p |= {n1 - 1, n1, n1 + 1, n - n1}
    p |= set(rng.integers(0, n, 48 if n <= 65536 else 16).tolist())
    return np.array(sorted(q for q in p if 0 <= q < n))


def tones(n, bins):
    k = np.arange(n)
    return np.stack([np.exp(2j * np.pi * ((b * k) % n) / n) for b in bins]).astype(np.complex64).ravel()


SPECIALS = ("zero", "subnormal", "up60", "down60", "inf", "nan")


def mixed(rng, n, frames, boundaries):
    """random dense frames; the special frames sit on both sides of each boundary (frame b - 1 and b), cycling through
    SPECIALS so that each kind meets several boundaries"""
    x = rnd_c32(rng, frames * n).reshape(frames, n)
    slots = sorted({f for b in boundaries for f in (b - 1, b) if 0 <= f < frames})
    for i, f in enumerate(slots):
        kind = SPECIALS[i % len(SPECIALS)]
        if kind == "zero":
            x[f] = 0
        elif kind == "subnormal":
            x[f] *= np.float32(2.0 ** -140)
        elif kind == "up60":
            x[f] *= np.float32(2.0 ** 60)
        elif kind == "down60":
            x[f] *= np.float32(2.0 ** -60)
        else:
            x[f, rng.integers(0, n)] = np.inf if kind == "inf" else np.nan
    return x.ravel()


def run_all(cb, n, inverse, rng, what, frame_counts, bounds_of, n1=None, path=None):
    """impulses, tones and the mixed batches of every frame count, one handle"""
    node = cb.FFTBatchNode(n, inverse)
    pos = impulse_positions(n, rng, n1)
    per = max(1, (1 << 23) // n)
    for i in range(0, len(pos), per):
        x = impulses(n, pos[i:i + per])
        check(node.run(x), x, n, inverse, what + " impulses", path)
    x = tones(n, sorted({1, 3, n // 4 + 1, n // 2 - 1, n - 5, (5 * n) // 7} - {0} if n > 1 else {0}))
    check(node.run(x), x, n, inverse, what + " tones", path)
    for frames in frame_counts:
        x = mixed(rng, n, frames, bounds_of(frames))
        check(node.run(x), x, n, inverse, f"{what} mixed x{frames}", path)


def child(env, jobs):
    """run jobs [(kind, args..., x)] in a child interpreter with `env` set (switches read once per process); returns
    their outputs.  kind 'fft': (n, inverse); 'fir': (taps, call sizes)"""
    code = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1])
import comms_rs_b200 as cb
cb.init(0)
d = np.load(sys.argv[2], allow_pickle=True)
out = {}
for i, job in enumerate(d["jobs"]):
    if job[0] == "fft":
        out[str(i)] = cb.FFTBatchNode(int(job[1]), bool(job[2])).run(job[3])
    else:
        node, x, pos, ys = cb.BatchFirNode(job[1]), job[3], 0, []
        for s in job[2]:
            ys.append(node.run(x[pos:pos + s]))
            pos += s
        out[str(i)] = np.concatenate(ys)
np.savez(sys.argv[3], **out)
"""
    with tempfile.TemporaryDirectory() as td:
        arr = np.empty(len(jobs), object)
        for i, j in enumerate(jobs):
            arr[i] = tuple(j)
        np.savez(os.path.join(td, "in.npz"), jobs=arr)
        subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(td, "in.npz"), os.path.join(td, "out.npz")],
                       check=True, env=dict(os.environ, **env), timeout=600)
        with np.load(os.path.join(td, "out.npz")) as r:
            return [r[str(i)] for i in range(len(jobs))]


# ------------------------------------------------------------------ direct O(N^2) sizes
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 10, 12, 100, 127])
@pytest.mark.parametrize("inverse", [False, True])
def test_direct_sizes(cb, n, inverse):
    # dft_direct_kernel: a grid-stride loop of 148 * 8 CTAs over the frames
    rng = np.random.default_rng(n * 2 + inverse)
    run_all(cb, n, inverse, rng, "direct", [7, 1185], lambda f: [1, 2, 1184] if f > 1000 else [1, 3, 6])


@pytest.mark.parametrize("n", [1000, 4095])
def test_direct_forced_up_to_4096(cb, n, monkeypatch):
    monkeypatch.setenv("COMMS_B200_FFT_PATH", "direct")
    rng = np.random.default_rng(n)
    for inverse in (False, True):
        node = cb.FFTBatchNode(n, inverse)
        x = np.concatenate([impulses(n, [0, 1, n // 2, n - 1]), mixed(rng, n, 8, [2, 6])])
        check(node.run(x), x, n, inverse, "direct forced", "direct")


# ------------------------------------------------------------------ one CTA per frame (or several frames per CTA)
@pytest.mark.parametrize("log2n", list(range(3, 15)))
@pytest.mark.parametrize("inverse", [False, True])
def test_single_cta_sizes(cb, log2n, inverse):
    n = 1 << log2n
    per = max(1, 4096 // n)  # frames per CTA (fft2_small_frames_kernel / fft2_frames_kernel)
    rng = np.random.default_rng(log2n * 2 + inverse)
    counts = [1, per + 1, 5 * per + 3] if n >= 1024 else [per - 1 if per > 1 else 1, 5 * per + 3]
    run_all(cb, n, inverse, rng, "single-cta", counts, lambda f: [per * i for i in range(1, f // per + 1)][:8])


@pytest.mark.parametrize("n", [16, 32, 64, 128])
def test_small_sizes_generic_kernel(cb, n, monkeypatch):
    monkeypatch.setenv("COMMS_B200_FFT_SMALL", "generic")
    rng = np.random.default_rng(n + 7)
    per = 4096 // n
    for inverse in (False, True):
        run_all(cb, n, inverse, rng, "generic-small", [3 * per + 1], lambda f: [per, 2 * per, 3 * per])


@pytest.mark.parametrize("n", [8192, 16384])
def test_8192_16384_two_level_kernel(cb, n, monkeypatch):
    monkeypatch.setenv("COMMS_B200_FFT_8K16K", "two")
    rng = np.random.default_rng(n + 9)
    for inverse in (False, True):
        run_all(cb, n, inverse, rng, "two-level", [13], lambda f: [1, 4, 8, 12], n1=256)


# ------------------------------------------------------------------ two-step splits, 2^15 .. 2^20
def _ring(n):
    return (48 << 20) // (8 * n)  # scratch_frames of the plan (cb_fft_create)


@pytest.mark.parametrize("log2n", list(range(15, 21)))
@pytest.mark.parametrize("path", ["default", "fourstep"])
def test_two_step_sizes(cb, log2n, path, monkeypatch):
    # default: the fused two-step kernel with its L2 ring (65536: the rows kernel); fourstep: the column-batch step
    # kernels in groups of ring frames (65536 points keep the rows kernel)
    n = 1 << log2n
    if path != "default":
        monkeypatch.setenv("COMMS_B200_FFT_PATH", path)
    ring = _ring(n)
    n1 = 1 << (log2n // 2)
    rng = np.random.default_rng(log2n * 3 + (path == "fourstep"))
    cap = max(2, min(ring + 2, (1 << 23) // n))  # frames per batch: past the ring where the reference allows
    counts = sorted({1, 2, ring // 2, min(ring, cap), cap})  # below, at and past the lag (ring / 2) and the ring
    for inverse in (False, True):
        run_all(cb, n, inverse, rng, f"two-step {path}", counts if inverse else counts[-1:],
                lambda f: [1, ring, f - 1], n1=n1)


@pytest.mark.parametrize("path", ["cluster", "cluster2", "cluster16", "twopass", "rows", "rows2", "big", "cpipe",
                                  "rowspf"])
def test_65536_paths(cb, path, monkeypatch):
    # every value of COMMS_B200_FFT_PATH that cb_fft_create maps to its own 65536-point kernel: clusters of 8 CTAs with
    # two exchange synchronisations and of 16 CTAs, the 16 x 4096 two-pass form, the ring of 96 frames (rows, rowspf),
    # its two-launch form, the generic fused two-step kernel and the pipelined clusters.  (Other values, fourstep
    # included, select the rows kernel at this size.)
    monkeypatch.setenv("COMMS_B200_FFT_PATH", path)
    n = 65536
    rng = np.random.default_rng(sum(map(ord, path)))
    for inverse in (False, True):
        counts = [1, 97] if path in ("rows", "rowspf", "rows2", "twopass") and inverse else [19]
        run_all(cb, n, inverse, rng, f"65536 {path}", counts, lambda f: [1, 8, 16, 96, f - 1], n1=256)


@pytest.mark.parametrize("env", [{"COMMS_B200_FFT_BIG_NT": "256"}, {"COMMS_B200_FFT_BIG_NT": "512"},
                                 {"COMMS_B200_FFT_BIG_NT": "1024"}, {"COMMS_B200_FFT_CTAS": "5"},
                                 {"COMMS_B200_FFT_CTAS": "6"}], ids=lambda e: "-".join(f"{k[12:]}={v}" for k, v in e.items()))
def test_two_step_process_switches(env):
    # threads per two-step kernel, CTAs per SM of the ring kernels: read once per process
    rng = np.random.default_rng(len(str(env)))
    jobs = []
    for log2n in (15, 17, 20) if "COMMS_B200_FFT_BIG_NT" in env else (16,):
        n = 1 << log2n
        frames = min(_ring(n) + 1, (1 << 22) // n)
        x = np.concatenate([impulses(n, impulse_positions(n, rng, 1 << (log2n // 2))[::4][:(1 << 23) // n]),
                            mixed(rng, n, frames, [1, frames - 1])])
        jobs += [("fft", n, False, x), ("fft", n, True, x)]
    for job, got in zip(jobs, child(env, jobs)):
        check(got, job[3], job[1], job[2], f"two-step {env}")


# ------------------------------------------------------------------ chirp-z
@pytest.mark.parametrize("n", [129, 1000, 4095, 4097, 8191, 10007, 65535, 300000])
@pytest.mark.parametrize("inverse", [False, True])
def test_chirpz(cb, n, inverse):
    # fused (M <= 16384: 4096 / M frames per CTA) and, above, the five-launch form around the two-step plans; both
    # reuse their work buffers per group of bl_frames, and every batch runs past the first group seam
    m = B.chirpz_m(n)
    group = max(1, ((32 if m <= 16384 else 256) << 20) // (m * 8))  # bl_frames (bluestein_setup)
    per = max(1, 4096 // m)
    rng = np.random.default_rng(n + inverse)
    frames = group + 2
    run_all(cb, n, inverse, rng, "chirp-z", [frames], lambda f: [per, 2 * per, group, f - 1])


def test_chirpz_split_form():
    rng = np.random.default_rng(11)
    jobs = []
    for n in (129, 1000, 4097, 8191):
        x = np.concatenate([impulses(n, [0, 1, n // 2, n - 1]), tones(n, [1, n // 3]), mixed(rng, n, 9, [2, 5, 8])])
        jobs += [("fft", n, False, x), ("fft", n, True, x)]
    for job, got in zip(jobs, child({"COMMS_B200_FFT_CHIRPZ": "split"}, jobs)):
        check(got, job[3], job[1], job[2], "chirp-z split")


# ------------------------------------------------------------------ overlap-save FIR
def _ols_case(ntaps, cplx, seed):
    rng = np.random.default_rng(300 + seed)
    t = rnd_c32(rng, ntaps) if cplx else rng.uniform(-1, 1, ntaps).astype(np.complex64)
    hop = B.OLS_N - (ntaps - 1)
    sizes = [8192, hop * 3, hop * 3 + 1, 100, 8191, 20_011, 8192 + hop - 1, 3]
    return t, sizes, rnd_c32(rng, sum(sizes))


def check_ols(got, x, t, sizes, what):
    """every output of every call: overlap-save calls (>= 8192 samples) against the OLS bound, seams first; the
    shorter calls (direct FIR) against tol * A_n"""
    K = len(t)
    pos, hist = 0, None
    for s in sizes:
        xs, gs = x[pos:pos + s], got[pos:pos + s]
        want, new_hist = B.fir64(xs, t, hist)
        if s >= 8192:
            bound, _ = B.ols_bound(xs, t, hist)
            err = np.abs(gs.astype(np.complex128) - want)
            seams = B.ols_seams(s, K)
            bad = seams[~(err[seams] <= bound[seams])]
            assert not len(bad), (f"{what}: call at {pos} ({s} samples): seam outputs {bad[:8].tolist()} outside the "
                                  f"OLS bound, |err|/bound = {(err[bad] / bound[bad])[:8]}")
            r = err / bound
            bad = np.flatnonzero(~(r <= 1))
            assert not len(bad), f"{what}: call at {pos}: outputs {bad[:8].tolist()} outside, ratio {r[bad[:8]]}"
            print(f"RATIO ols {what} call={s} worst={r.max():.4f}")
        else:
            B.assert_fir_bound(gs, want, B.fir_mag64(xs, t, hist), 1e-5, f"{what}: direct call at {pos}")
        hist = new_hist
        pos += s


@pytest.mark.parametrize("ntaps", [129, 500, 1024, 1025])
@pytest.mark.parametrize("cplx", [False, True])
def test_overlap_save_fused(cb, ntaps, cplx):
    t, sizes, x = _ols_case(ntaps, cplx, ntaps + cplx)
    node, pos, outs = cb.BatchFirNode(t), 0, []
    for s in sizes:
        outs.append(node.run(x[pos:pos + s]))
        pos += s
    check_ols(np.concatenate(outs), x, t, sizes, f"fused K={ntaps} cplx={cplx}")


def test_overlap_save_split():
    jobs = []
    for ntaps, cplx in ((129, True), (500, False), (1024, True), (1025, False)):
        t, sizes, x = _ols_case(ntaps, cplx, ntaps + cplx)
        jobs.append(("fir", t, sizes, x))
    for job, got in zip(jobs, child({"COMMS_B200_FIR_OLS": "split"}, jobs)):
        check_ols(got, job[3], job[1], job[2], f"split K={len(job[1])}")


@pytest.mark.parametrize("ntaps", [129, 1025])
def test_overlap_save_inf_stays_in_its_frames(cb, ntaps):
    # one Inf sample: the outputs of exactly the frames whose 4096 inputs hold it are non-finite, all others finite and
    # within the bound
    rng = np.random.default_rng(ntaps)
    t = rnd_c32(rng, ntaps)
    hop = B.OLS_N - (ntaps - 1)
    n = 6 * hop + 77
    x = rnd_c32(rng, n)
    j = 3 * hop + 5  # inside frame 3, and in frame 4's history when the taps are long
    x[j] = np.inf
    got = cb.BatchFirNode(t).run(x)
    f = np.arange(n) // hop
    holds = (f * hop - (ntaps - 1) <= j) & (j < f * hop - (ntaps - 1) + B.OLS_N)
    fin = np.isfinite(got.real) & np.isfinite(got.imag)
    assert np.array_equal(~fin, holds), (np.flatnonzero(~fin)[:5], np.flatnonzero(holds)[:5])
    xc = x.copy()
    xc[j] = 0  # the bound of the clean frames does not involve the Inf
    want, _ = B.fir64(xc, t)
    bound, _ = B.ols_bound(xc, t)
    err = np.abs(got[fin].astype(np.complex128) - want[fin])
    assert np.all(err <= bound[fin]), (err / bound[fin]).max()
