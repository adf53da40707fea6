"""CPU-only checks of the boundary and host logic: the C-ABI library loads and
exports exactly what include/comms_b200.h declares, fails loudly without a GPU,
and the multi-GPU partitioning (world_size 2, gloo) reproduces the one-shot result."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cb():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge

    ge._load_build_module().build()
    import comms_rs_b200 as m

    return m


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "comms_b200.h")).read()
    return sorted(set(re.findall(r"CB_API[^;(]*?\b(cb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol(cb):
    lib = cb.load()
    names = _header_symbols()
    assert len(names) >= 50
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/comms_b200.h but not exported"
    assert sorted(cb._lib.SIGNATURES) == names  # the binding covers the header, no more, no less
    out = subprocess.run(["nm", "-D", "--defined-only", cb._lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(s for s in re.findall(r" T (\w+)", out) if s.startswith("cb_"))
    assert exported == names  # nothing else leaks out of the .so


def test_rust_shim_sources_track_the_library(cb):
    # the Rust crate cannot be compiled in this image; keep its hand-written parts honest at least: build.rs compiles
    # the same sources as build.py, and ffi.rs declares every entry of the header (and nothing that does not exist)
    import importlib.util

    spec = importlib.util.spec_from_file_location("_cb_build", os.path.join(ROOT, "comms-rs_b200", "build.py"))
    bld = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bld)
    rs = open(os.path.join(ROOT, "comms-rs_b200", "rust", "build.rs")).read()
    assert sorted(set(re.findall(r'"(\w+\.cu)"', rs))) == sorted(bld.SOURCES)
    ffi = open(os.path.join(ROOT, "comms-rs_b200", "rust", "src", "ffi.rs")).read()
    assert sorted(set(re.findall(r"pub fn (cb_\w+)\(", ffi))) == _header_symbols()


def test_every_header_entry_cites_the_reference():
    src = open(os.path.join(ROOT, "include", "comms_b200.h")).read()
    for cite in ("src/filter/fir.rs:87-102", "src/util/resample_node.rs:53-65", "src/mixer.rs:43-51",
                 "src/fft/mod.rs:73-96", "src/modulation/analog.rs:22-34", "src/pulse.rs:82-92", "src/prns.rs:64-71"):
        assert cite in src


def test_no_device_fails_loudly_no_fallback(cb):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert cb.device_count() == 0
    with pytest.raises(cb.CbError) as e:
        cb.init(0)
    assert e.value.status == cb._lib.CB_ERR_NO_DEVICE and "no CPU fallback" in str(e.value)
    for ctor in (lambda: cb.BatchFirNode(np.ones(4, np.complex64)), lambda: cb.MixerNode(0.1),
                 lambda: cb.FFTBatchNode(1024), lambda: cb.FMDemodNode(),
                 lambda: cb.ChainBank(2, np.ones(4, np.complex64), 2), lambda: cb.DecimateNode(2).run(np.arange(4))):
        with pytest.raises((cb.CbError, cb.NodeError)):
            ctor()


def test_status_strings_and_version(cb):
    lib = cb.load()
    assert lib.cb_version() >= 1
    assert lib.cb_status_str(0) == b"ok" and lib.cb_status_str(2) == b"size mismatch"
    assert cb.launch_count() == 0 or cb.launch_count() > 0


def test_rrc_taps_host_entry(cb, oracle):
    # cb_rrc_taps restates rrc_taps (src/util/math.rs:221-280) on the host side of the C ABI; it needs no
    # device.  Golden vector math.rs:359-401, the config banks, and the oracle bit for bit.
    from golden import reference_vectors as G

    rrc = cb.rrc_taps(33, 3.18, 0.234, dtype=np.complex128)
    assert np.all(np.abs(rrc - np.array(G.RRC_33)) < np.finfo(np.float32).eps) and np.all(rrc.imag == 0)
    for n, sps, beta in [(32, 4.0, 0.25), (64, 4.0, 0.25), (1024, 8.0, 0.25), (33, 3.18, 0.234), (17, 4.0, 0.0),
                         (9, 4.0, 1.0), (41, 4.0, 0.5), (1, 2.0, 0.3), (0, 2.0, 0.3)]:
        for dt in (np.complex64, np.complex128):
            assert cb.rrc_taps(n, sps, beta, dtype=dt).tobytes() == oracle.rrc_taps(n, sps, beta, dtype=dt).tobytes()
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError):
            cb.rrc_taps(8, 4.0, bad)


def test_qfilt_taps_host_entry(cb, oracle):
    # cb_qfilt_taps_f64 restates qfilt_taps (src/util/math.rs:307-342) on the host side of the C ABI (no device): the
    # oracle bit for bit, including the L'Hospital branch (|2 alpha t| == 1) and the even -> odd length rule
    for n, alpha, sps in [(21, 0.25, 2), (101, 0.5, 10), (20, 0.25, 2), (33, 0.234, 3), (9, 1.0, 2), (5, 0.0, 4), (65, 0.5, 4),
                          (1, 0.3, 2)]:
        a, b = cb.qfilt_taps(n, alpha, sps), oracle.qfilt_taps(n, alpha, sps)
        assert len(a) == (n if n % 2 else n + 1) and a.tobytes() == np.asarray(b, np.float64).tobytes()
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError):
            cb.qfilt_taps(9, bad, 2)


def test_product_never_touches_the_oracle():
    # only tests/, __graft_entry__.smoke() and bench.py's CPU legs may use oracle/
    pkg = os.path.join(ROOT, "comms-rs_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp", ".rs")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "oracle" not in txt.lower() or f in ("misc_kernels.cu",), os.path.join(dp, f)


def test_segment_bounds_and_halo(cb):
    sh = cb.sharding
    for total, world, mult in [(1 << 20, 8, 1), (1000, 3, 10), (7, 8, 1), (100, 4, 7)]:
        segs = [sh.segment_bounds(total, world, r, mult) for r in range(world)]
        assert segs[0][0] == 0 and segs[-1][1] == total
        for (a, b), (c, d) in zip(segs, segs[1:]):
            assert b == c and a % mult == 0 and c % mult == 0
    assert [sh.block_shard(10, 4, r) for r in range(4)] == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert sh.halo_state(np.array([1, 2, 3], np.complex64), 5).tolist() == [3, 2, 1, 0, 0]
    assert sh.halo_state(np.array([1, 2, 3, 4], np.complex64), 2).tolist() == [4, 3]


_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["CB_ROOT"])
import numpy as np, torch, torch.distributed as dist
import comms_rs_b200 as cb, oracle
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
sh = cb.sharding
total, K, D = 50_000, 64, 10
x = oracle.synth_uniform_c32(5, 0, total)
taps = oracle.rrc_taps(K, 4.0, 0.25)
dphase, phase0 = 0.3711, 0.25
# (1) long stream, segment + halo: mixer -> FIR -> decimate, then ordered gather
a, b = sh.segment_bounds(total, world, rank, D)
mix = oracle.Mixer(sh.segment_phase(phase0, dphase, a), dphase)
lo = max(a - K, 0)
pre = oracle.Mixer(sh.segment_phase(phase0, dphase, lo), dphase).mix(x[lo:a]) if a > lo else np.zeros(0, np.complex64)
y, _ = oracle.batch_fir(mix.mix(x[a:b]), taps, sh.halo_state(pre, K))
y = oracle.decimate(y, D)
sizes = [len(range(*sh.segment_bounds(total, world, r, D))) for r in range(world)]
sizes = [-(-s // D) for s in sizes]
full = sh.gather_ordered(torch.from_numpy(y), sizes).numpy()
ref, _ = oracle.batch_fir(oracle.Mixer(phase0, dphase).mix(x), taps, np.zeros(K, np.complex64))
ref = oracle.decimate(ref, D)
assert full.shape == ref.shape
err = np.linalg.norm(full - ref) / np.linalg.norm(ref)
assert err < 1e-6, err   # only the mixer phase at the segment start differs (f64 rounding)
# without the mixer the segments are bit-exact
y2, _ = oracle.batch_fir(x[a:b], taps, sh.halo_state(x[lo:a], K))
full2 = sh.gather_ordered(torch.from_numpy(y2), [len(range(*sh.segment_bounds(total, world, r, D))) for r in range(world)]).numpy()
ref2, _ = oracle.batch_fir(x, taps, np.zeros(K, np.complex64))
assert full2.tobytes() == ref2.tobytes()
# (2) independent channels: block shard, no exchange needed for compute
c0, c1 = sh.block_shard(6, world, rank)
assert (c1 - c0) == 3
# (3) batched FFT: frames block-sharded, ordered gather = the transform of the whole batch, bit for bit
N, frames = 256, 11
f0, f1 = sh.block_shard(frames, world, rank)
xf = oracle.synth_uniform_c32(9, 0, frames * N)
yf = oracle.fft(xf[f0 * N:f1 * N], N, False)
fsz = [N * len(range(*sh.block_shard(frames, world, r))) for r in range(world)]
assert sh.gather_ordered(torch.from_numpy(yf), fsz).numpy().tobytes() == oracle.fft(xf, N, False).tobytes()
# (4) the real second stage of fm_radio (Complex(x, 0) -> FIR -> .re -> /5): segments on the decimation grid, halo as state
xr = oracle.synth_uniform_c32(11, 0, total).real.copy()
a5, b5 = sh.segment_bounds(total, world, rank, 5)
lo5 = max(a5 - K, 0)
y5, _ = oracle.batch_fir(xr[a5:b5].astype(np.complex64), taps, sh.halo_state(xr[lo5:a5].astype(np.complex64), K))
y5 = oracle.decimate(y5.real.copy(), 5)
sz5 = [-(-len(range(*sh.segment_bounds(total, world, r, 5))) // 5) for r in range(world)]
ref5, _ = oracle.batch_fir(xr.astype(np.complex64), taps, np.zeros(K, np.complex64))
assert sh.gather_ordered(torch.from_numpy(y5), sz5).numpy().tobytes() == oracle.decimate(ref5.real.copy(), 5).tobytes()
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_two_rank_gloo_segment_sharding(cb, oracle, tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, CB_ROOT=ROOT, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("ok") == 2


def test_bench_reference_arm_prints_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--workload", "fft1024"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Msamples/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_rejects_arguments_it_would_not_honour(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr, (extra, r.stderr[-2000:])
    assert not (tmp_path / "d").exists()


def test_bench_dump_sample_is_fixed_and_covers_the_output():
    import importlib.util

    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.sample_rows(1000, 1000) is None
    for rows, k in ((1 << 28, 1 << 23), (1001, 1000), (13421773, 777)):
        idx = bench.sample_rows(rows, k)
        assert len(idx) == k and idx.tobytes() == bench.sample_rows(rows, k).tobytes()
        stride = rows // k
        assert np.array_equal(idx // stride, np.arange(k)) and idx[-1] < rows  # one row in each stratum, in order


def test_bench_cpu_leg_runs_for_every_workload_kind():
    # the reference arm / cpu_baseline leg of bench.py for one workload of every kind, on a small sample
    import importlib.util

    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    kinds = {}
    for name, (kind, *_rest) in bench.WORKLOADS.items():
        kinds.setdefault(kind, name)
    assert set(kinds) == {"fir", "fir16", "fft16", "firdec", "firreal", "graph", "fft", "est", "mixer", "fm", "chain", "interp"}
    for kind, name in kinds.items():
        rate, dt, n = bench.cpu_rate(name, 1 << 15, 2)
        assert rate > 0 and n > 0, name
    rate, _, _ = bench.cpu_rate("timing10x5", 1 << 14, 1)
    assert rate > 0


@pytest.mark.parametrize("D", [2, 4, 5, 8, 10])
def test_real_fir_kernel_index_algebra(D, oracle):
    # The polyphase bookkeeping of fir_real_decim_kernel<D> (csrc/fir_real_kernel.cu), restated index for index in numpy:
    #   A_p[i] = x[(J0 - LB + i) D - p]  filled from the linear range g = G0 + e with i = e / D, p = D - 1 - e % D,
    #   thread t / output u reads w[u - q + LB] = A_p[4 t + u - q + LB]  for tap k = q D + p.
    # It must reproduce y[J] = sum_k h[k] x[J D - k] (history for negative indices) -- checked against the oracle.
    rng = np.random.default_rng(D)
    NT, TO = 256, 1024
    Q = (64 + D - 1) // D
    LB = (Q - 1 + 3) // 4 * 4
    LEN = TO + LB
    ntaps, H = 63, 64
    h = rng.uniform(-1, 1, ntaps).astype(np.float32)
    n_in = 2 * TO * D + 3 * D + 1  # two full tiles and a ragged third
    x = rng.uniform(-1, 1, n_in).astype(np.float32)
    hist = rng.uniform(-1, 1, H).astype(np.float32)  # chronological, hist[H - 1] = x[-1]
    n_out = -(-n_in // D)
    taps = np.zeros(80, np.float32)
    taps[:ntaps] = h

    def sample(g):
        if g >= 0:
            return x[g] if g < n_in else np.float32(0)
        return hist[H + g] if g + H >= 0 else np.float32(0)

    y = np.zeros(n_out, np.float64)
    for tile in range(-(-n_out // TO)):
        J0 = tile * TO
        G0 = (J0 - LB) * D - (D - 1)
        A = np.zeros((D, LEN), np.float64)
        for e in range(LEN * D):
            A[D - 1 - e % D, e // D] = sample(G0 + e)
        for t in range(NT):
            for u in range(4):
                J = J0 + 4 * t + u
                if J >= n_out:
                    continue
                acc = 0.0
                for p in range(D):
                    w = A[p, 4 * t:4 * t + LB + 4]
                    for q in range(Q):
                        if q * D + p < 64:
                            acc += float(taps[q * D + p]) * w[u - q + LB]
                y[J] = acc
    state = np.concatenate([hist[::-1], np.zeros(max(0, ntaps - H))]).astype(np.complex64)[:ntaps]
    full, _ = oracle.batch_fir(x.astype(np.complex64), h.astype(np.complex64), state)
    want = oracle.decimate(full.real.copy(), D)
    assert y.shape == want.shape
    assert np.linalg.norm(y - want) <= 1e-6 * np.linalg.norm(want)


@pytest.mark.parametrize("ntaps", [1, 3, 5, 21, 101, 103])
def test_timing_kernel_window_algebra(ntaps):
    # The shared-memory geometry of timing_partial_kernel (csrc/estimator_kernels.cu: timing_geo, the mod-4
    # de-interleaved tile, the 7-sample sliding register window, four taps per step), restated index for index:
    # it must give y[i] = sum_k h[k] q[i - k] for every output of a tile, whatever ntaps mod 4 is.
    rng = np.random.default_rng(ntaps)
    NT, TILE = 256, 1024
    halo = ntaps - 1
    ntaps4 = (ntaps + 3) & ~3
    lead = 4 + ((4 - halo % 4) % 4)
    h4 = halo + lead
    assert h4 % 4 == 0 and 4 <= lead <= 7
    pitch = (TILE + h4) // 4
    while pitch % 8 != 2:
        pitch += 1
    taps = np.zeros(ntaps4)
    taps[:ntaps] = rng.uniform(-1, 1, ntaps)
    n = 2 * TILE + 37
    q = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    want = np.convolve(q, taps[:ntaps])[:n]
    for tile in range(-(-n // TILE)):
        i0 = tile * TILE
        sm = np.full(4 * pitch, np.nan + 0j)  # anything not written must not be used with a non-zero tap
        for e in range(TILE + h4):
            m = i0 - h4 + e
            sm[(e & 3) * pitch + (e >> 2)] = q[m] if (e >= lead and 0 <= m < n) else 0.0
        for t in range(NT):
            c = [(h4 >> 2) + t + k * pitch for k in range(4)]  # class k: L[base + k]
            W = [sm[c[1] - 1], sm[c[2] - 1], sm[c[3] - 1], sm[c[0]], sm[c[1]], sm[c[2]], sm[c[3]]]
            y = [0j] * 4
            for k in range(0, ntaps4, 4):
                for u in range(4):
                    for r in range(4):
                        if taps[k + r] != 0.0:
                            y[u] += taps[k + r] * W[u - r + 3]
                back = (k >> 2) + 1
                idx = [c[1] - 1 - back, c[2] - 1 - back, c[3] - 1 - back, c[0] - back]
                W = [sm[j] if 0 <= j < len(sm) else np.nan for j in idx] + W[:3]
            for u in range(4):
                i = i0 + 4 * t + u
                if i < n:
                    assert abs(y[u] - want[i]) <= 1e-12 * (1 + abs(want[i])), (tile, t, u)


@pytest.mark.parametrize("L1,L2", [(7, 8), (8, 8), (8, 9), (9, 9)])
def test_two_step_fft_split_algebra(L1, L2):
    # the N1 x N2 split of fft_big_kernel.cu / fft_rows_kernel.cu: n = N2 n1 + n2, k = k1 + N1 k2,
    # X[k1 + N1 k2] = sum_n2 W_N2^{n2 k2} { W_N^{n2 k1} sum_n1 x[N2 n1 + n2] W_N1^{n1 k1} }
    N1, N2 = 1 << L1, 1 << L2
    N = N1 * N2
    rng = np.random.default_rng(L1 * 16 + L2)
    x = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    for inverse in (False, True):
        sgn = 1.0 if inverse else -1.0
        f = (lambda a, axis: np.fft.ifft(a, axis=axis) * a.shape[axis]) if inverse else (lambda a, axis: np.fft.fft(a, axis=axis))
        Y = f(x.reshape(N1, N2), 0)                                   # step A: [k1][n2], stored in place
        k1, n2 = np.meshgrid(np.arange(N1), np.arange(N2), indexing="ij")
        Z = Y * np.exp(sgn * 2j * np.pi * (k1 * n2 % N) / N)          # twiddle on the way into step B
        X = f(Z, 1)                                                   # step B: rows; X[k1 + N1 k2]
        got = X.T.reshape(-1)                                         # index k1 + N1 k2 -> k2-major
        want = f(x, 0)
        assert np.linalg.norm(got - want) <= 1e-11 * np.linalg.norm(want)


@pytest.mark.parametrize("L2", [5, 6])
def test_two_level_fft_layout_is_conflict_free_and_covers_the_frame(L2):
    # fft2_two_level_kernel (fft_kernels.cu), 8192 / 16384 points = 256 x N2: element (b, a) of the transposed frame lives
    # at rb(b) + pad16(a) with rb(b) = b * 304 + b // T2 + (16 // T2) * (b % T2).  (1) no two elements share a word;
    # (2) the 16 lanes of a half-warp hit 16 different 8-byte banks in all three access patterns: the transposing store
    # (b = 2 i resp. 2 i + 1, a fixed), the row accesses of level 1 (positions 17 m + j and 17 j + q of one row) and the
    # column accesses of level 2 (k1 = k0 .. k0 + 16 / T2 - 1, b = j2 + T2 m, j2 < T2).
    N2 = 1 << L2
    T2, RP = N2 // 16, 304
    pad16 = lambda i: i + (i >> 4)
    rb = lambda b: b * RP + b // T2 + (16 // T2) * (b % T2)
    cells = {rb(b) + pad16(a) for b in range(N2) for a in range(256)}
    assert len(cells) == N2 * 256 and max(cells) < N2 * RP  # injective, inside the buffer (the table follows it)
    bank = lambda addr: addr % 16
    for a in (0, 1, 15, 16, 255):
        for half in range(N2 // 32 if N2 >= 32 else 1):
            for odd in (0, 1):
                lanes = [rb(2 * i + odd + 32 * half) + pad16(a) for i in range(16)]
                assert len({bank(x) for x in lanes}) == 16
    for b in (0, 1, N2 - 1):
        for m in range(16):
            assert len({bank(rb(b) + pad16(j + 16 * m)) for j in range(16)}) == 16
        for q in range(16):
            assert len({bank(rb(b) + pad16(16 * j + q)) for j in range(16)}) == 16
    per = 16 // T2
    for k0 in range(0, 256, per):
        for m in range(16):
            lanes = [rb(j2 + T2 * m) + pad16(k0 + i) for i in range(per) for j2 in range(T2)]
            assert len({bank(x) for x in lanes}) == 16, (k0, m)
    # and the algebra: X[k1 + 256 k2] = sum_b W_N2^{b k2} { W_N^{b k1} sum_a x[N2 a + b] W_256^{a k1} }
    N = 256 * N2
    rng = np.random.default_rng(L2)
    x = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    Y = np.fft.fft(x.reshape(256, N2), axis=0)                       # rows b (columns of this view): Y[k1][b]
    k1, b = np.meshgrid(np.arange(256), np.arange(N2), indexing="ij")
    X = np.fft.fft(Y * np.exp(-2j * np.pi * (k1 * b) / N), axis=1)    # X[k1][k2]
    assert np.linalg.norm(X.T.reshape(-1) - np.fft.fft(x)) <= 1e-10 * np.linalg.norm(x) * np.sqrt(N)


@pytest.mark.parametrize("log2n", [4, 5, 6, 7])
def test_small_fft_staging_is_warp_local(log2n):
    # fft2_small_frames_kernel: warp w of the CTA stages points [512 w, 512 w + 512) of the CTA's 4096, thread t transforms
    # frame t // T with T = N / 16 threads per frame.  The frames a warp's threads transform must be exactly the frames
    # whose points that warp staged (so that warp barriers suffice), and a pair of points loaded together never
    # straddles two frames.
    N = 1 << log2n
    T = N // 16
    for w in range(8):
        staged = {i >> log2n for i in range(512 * w, 512 * w + 512)}
        transformed = {t // T for t in range(32 * w, 32 * w + 32)}
        assert staged == transformed
    assert all((i >> log2n) == ((i + 1) >> log2n) for i in range(0, 4096, 2))


@pytest.mark.parametrize("nframes,ring,ctas", [(40, 8, 3), (200, 96, 592), (9, 4, 1), (64, 16, 7)])
def test_fused_fft_held_tickets_cannot_deadlock(nframes, ring, ctas):
    # the 65536-point kernels of this round hold tickets ahead of the item they run: K5-R one (requested at the top of an
    # item), K5-R2 two, and both release an item's counter only at the top of the NEXT item.  Simulate `ctas` CTAs with
    # a two-ticket look-ahead and the deferred release: a CTA runs its item only when the item's dependency counter is
    # complete; every schedule in which CTAs are picked round-robin must finish all items (no deadlock), because a CTA
    # never waits while it still owes a release.
    ITEMS = 16
    lag = max(ring // 2, 1)
    total = (lag + 2 * nframes) * ITEMS

    def decode(item):
        chunk = item // ITEMS
        if chunk < lag:
            return True, chunk
        t = chunk - lag
        return (t % 2 == 0), (lag + t // 2 if t % 2 == 0 else t // 2)

    done_a, done_b = [0] * nframes, [0] * nframes
    ticket = 0
    state = []
    for _ in range(ctas):  # each CTA: [current ticket, next ticket, owed release]
        state.append([ticket, ticket + 1, None])
        ticket += 2
    finished = 0
    idle_rounds = 0
    while finished < ctas:
        progressed = False
        for st in state:
            if st[0] is None:
                continue
            if st[2] is not None:  # top of an item: pay the previous item's release first
                is_a, f = st[2]
                (done_a if is_a else done_b)[f] += 1
                st[2] = None
                progressed = True
            if st[0] >= total:
                st[0] = None
                finished += 1
                progressed = True
                continue
            is_a, f = decode(st[0])
            if f < nframes:
                ready = (done_a[f] == ITEMS) if not is_a else (f < ring or done_b[f - ring] == ITEMS)
                if not ready:
                    continue  # blocking wait; nothing is owed
                st[2] = (is_a, f)
            st[0], st[1] = st[1], ticket
            ticket += 1
            progressed = True
        idle_rounds = 0 if progressed else idle_rounds + 1
        assert idle_rounds < 2, "deadlock"
    assert all(v == ITEMS for v in done_a) and all(v == ITEMS for v in done_b)


@pytest.mark.parametrize("nframes,ring", [(1, 4), (5, 4), (33, 32), (100, 8), (7, 2)])
def test_fused_fft_ticket_order_cannot_wait_on_a_later_ticket(nframes, ring):
    # the work order of the fused two-step FFT kernels: A(0 .. lag-1), then A(lag + u), B(u) alternating, ITEMS items per
    # (frame, step), handed out by one ticket counter.  An item waits for: B(f) on all A(f) items; A(f >= ring) on all
    # B(f - ring) items.  Every such dependency must carry a SMALLER ticket -- then the earliest unfinished item can
    # always run and the kernel cannot deadlock however few CTAs are resident.
    ITEMS = 8
    lag = max(ring // 2, 1)
    nchunks = lag + 2 * nframes
    first, last = {}, {}
    for item in range(nchunks * ITEMS):
        chunk = item // ITEMS
        if chunk < lag:
            is_a, frame = True, chunk
        else:
            t = chunk - lag
            is_a = t % 2 == 0
            frame = lag + t // 2 if is_a else t // 2
        if frame >= nframes:
            continue
        key = ("A" if is_a else "B", frame)
        first.setdefault(key, item)
        last[key] = item
    assert sorted(first) == sorted([(s, f) for s in "AB" for f in range(nframes)])  # every (step, frame) exactly once
    for f in range(nframes):
        assert last[("A", f)] < first[("B", f)]
        if f >= ring:
            assert last[("B", f - ring)] < first[("A", f)]


def test_halo_state_for_polyphase_segments_matches_the_oracle_state(cb):
    # the reference `state` (src/filter/fir_node.rs:193-200) a rank hands to its polyphase bank: zero-stuffed domain, the
    # i-th most recent symbol at index i*L - 1.  Must equal the state the oracle's UpsampleNode -> batch_fir carries.
    import oracle

    rng = np.random.default_rng(5)
    for L, ntaps in ((8, 1024), (4, 32), (3, 17), (1, 64)):
        sym = (rng.uniform(-1, 1, 300) + 1j * rng.uniform(-1, 1, 300)).astype(np.complex64)
        taps = rng.uniform(-1, 1, ntaps).astype(np.complex64)
        _, st = oracle.batch_fir(oracle.upsample(sym, L) if L > 1 else sym, taps, np.zeros(ntaps, np.complex64))
        mine = cb.sharding.halo_state(sym, ntaps, L)
        if L == 1:
            assert mine.tobytes() == st.tobytes()
        else:
            # after the last stuffed zeros the reference state is shifted by L - 1 slots: entries that hold symbols agree
            k = np.arange(L - 1, ntaps, L)
            i = (k + 1) // L
            assert np.array_equal(mine[k], sym[len(sym) - i])
            assert np.count_nonzero(np.delete(mine, k)) == 0
        # segment = suffix: filtering the second half from that state reproduces the one-stream output exactly
        h = 150
        full, _ = oracle.batch_fir(oracle.upsample(sym, L) if L > 1 else sym, taps, np.zeros(ntaps, np.complex64))
        part, _ = oracle.batch_fir(oracle.upsample(sym[h:], L) if L > 1 else sym[h:], taps, cb.sharding.halo_state(sym[:h], ntaps, L))
        assert part.tobytes() == full[h * L:].tobytes()


def test_segment_phase_is_exact_for_long_streams(cb):
    # phase0 + start * dphase reduced exactly (ADVICE r01: a plain f64 product is 2e-6 rad off at 2^31 samples)
    from fractions import Fraction
    import math

    two_pi = Fraction("6.28318530717958647692528676655900576839433879875021")
    for phase0, dphase, start in ((0.1, 0.123, 5), (0.0, 6.2, (1 << 31) + 12345), (3.0, 0.7853981633974483, 1 << 40), (0.5, 1e-9, 1 << 33)):
        got = cb.sharding.segment_phase(phase0, dphase, start)
        p = Fraction(phase0) + Fraction(start) * Fraction(dphase)
        want = float(p - (p // two_pi) * two_pi)
        assert 0.0 <= got < 2 * math.pi
        assert abs(got - want) < 1e-15 or abs(abs(got - want) - 2 * math.pi) < 1e-12
    assert cb.sharding.segment_phase(0.25, 0.5, 0) == 0.25


def test_segment_bounds_cover_ragged_totals(cb):
    for total, world, mult in ((7344129, 8, 1 << 20), (10, 4, 4), (5, 8, 1), (1 << 28, 8, 10)):
        b = [cb.sharding.segment_bounds(total, world, r, mult) for r in range(world)]
        assert b[0][0] == 0 and b[-1][1] == total
        for (a0, a1), (b0, b1) in zip(b, b[1:]):
            assert a1 == b0 and a0 <= a1
        assert all(s % mult == 0 for s, _ in b if s < total)


def test_reference_arm_never_maps_the_product():
    # bench.py --impl reference times the oracle port only: neither the package nor libcomms_b200.so may be loaded
    import subprocess
    import sys

    code = (
        "import sys, runpy\n"
        "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '3', '--workload', 'pulse4']\n"
        f"runpy.run_path({os.path.join(ROOT, 'bench.py')!r}, run_name='__main__')\n"
        "maps = open('/proc/self/maps').read()\n"
        "assert 'libcomms_b200' not in maps and 'comms_rs_b200' not in sys.modules, 'product loaded by the reference arm'\n"
    )
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["gpu_launches"] == 0


def test_hot_kernels_keep_their_register_budgets_and_do_not_spill(cb):
    # the occupancies DESIGN.md quotes rest on register counts: 64 registers x 256 threads x 4 CTAs per SM for the
    # frame FFTs, 576 x 95 for the persistent tensor-core FIR, ... and on no local-memory spills.  Read them from the
    # built library (cuobjdump --dump-resource-usage) so that a compiler or source change that breaks one is seen on
    # the CPU box, not as a silent slowdown on the GPU.
    import re
    import shutil
    import subprocess

    # the cuobjdump of the toolkit build.py compiles with, which need not be on PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cuobjdump = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.dirname(nvcc))
    if cuobjdump is None:
        pytest.skip("cuobjdump not found on PATH or beside nvcc")
    lib = os.path.join(ROOT, "comms-rs_b200", "libcomms_b200.so")
    out = subprocess.run([cuobjdump, "--dump-resource-usage", lib], capture_output=True, text=True, check=True).stdout
    usage = {}
    for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+)", out):
        usage[m.group(1)] = (int(m.group(2)), int(m.group(3)))
    assert len(usage) > 100

    def find(*parts):
        hits = [(k, v) for k, v in usage.items() if all(p in k for p in parts)]
        assert hits, parts
        return hits

    budgets = [  # (name fragments, max registers, threads, CTAs per SM the launch code counts on, max stack bytes)
        (("fft2_frames_kernelILi12E",), 64, 256, 4, 0),
        (("fft2_frames_kernelILi10E",), 64, 256, 4, 0),
        (("fft2_small_frames_kernel",), 64, 256, 4, 0),
        (("fft65536_fused_kernel", "ELi4EEE"), 64, 256, 4, 0),
        (("fft65536_fused_kernel", "ELi5EEE"), 48, 256, 5, 0),
        (("fft65536_pf_kernel",), 72, 288, 3, 0),
        (("fft_big_fused_kernelILi7ELi8ELi256E",), 64, 256, 4, 0),
        (("fir_tc_kernelILi3ELi2E",), 112, 576, 1, 0),
        (("fir_ptc_kernel", "ELb0ELi"), 168, 320, 1, 0),   # f32 output: 4 epilogue warps
        (("fir_ptc_kernel", "ELb1ELi"), 144, 448, 1, 0),   # i16 output: 8 epilogue warps
        (("chain_tc_kernel",), 102, 640, 1, 0),
        (("chain3_kernelILb1ELb1ELb0ELi10ELi3ELi128ELi2ELi3E",), 136, 160, 3, 64),  # (a 32-byte local array, no spills)
    ]
    for parts, max_regs, threads, ctas, max_stack in budgets:
        for name, (regs, stack) in find(*parts):
            assert stack <= max_stack, (name, "stack", stack)
            assert regs <= max_regs, (name, regs)
            assert regs * threads * ctas <= 65536, (name, regs, threads, ctas)
