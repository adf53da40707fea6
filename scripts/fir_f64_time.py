"""Time the Complex<f64> FIR (BatchFirNodeF64.run_dev) with CUDA events on device-resident inputs, against an FP64 FMA
rate probe compiled and run in the same process (scripts/fp64_probe.cu).

    python scripts/fir_f64_time.py [--n-log2 26] [--reps 20] [--out results.jsonl]

Inputs are 2^n-log2 complex f64 samples (2^26: 1 GiB in, 1 GiB out, larger than L2) except for the x8 interpolator,
which takes 2^(n-log2 - 3) symbols so that it too writes 2^n-log2 samples.  Each shape is warmed up, then timed over
--reps calls: median and minimum.  Useful DFMA counts only the products the filter needs (4 per complex term, 2 per
real term; none with stuffed zeros).  Also timed, for context: the f32 BatchFirNode on the 64-complex-tap shape (the
price of f64) and the one-thread CPU oracle (orc_batch_fir_c64) on 2^20 samples.  Prints one JSON line per result,
the first with the card's name and power limit.  Writes nothing in the tree; the probe is built in a temporary
directory."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [  # name, taps, real, decim, interp
    ("64 real", 64, True, 1, 1),
    ("64 complex", 64, False, 1, 1),
    ("101 real (timing estimator)", 101, True, 1, 1),
    ("1025 complex", 1025, False, 1, 1),
    ("63 real /5", 63, True, 5, 1),
    ("1024 real x8 polyphase", 1024, True, 1, 8),
]


def time_events(torch, fn, stream, reps, warm=3):
    for _ in range(warm):
        fn()
    stream.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def taps_for(cb, k, real):
    t = cb.rrc_taps(k, 4.0, 0.25, dtype=np.complex128)
    return t if real else t * np.exp(0.1j * np.arange(k))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-log2", type=int, default=26)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    import comms_rs_b200 as cb
    import oracle

    cb.init(0)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    emit({"what": "device", "gpu": gpu, "torch_name": torch.cuda.get_device_name(0)})
    s = torch.cuda.Stream()

    # FP64 FMA rate of independent chains
    with tempfile.TemporaryDirectory() as td:
        so = os.path.join(td, "fp64_probe.so")
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler", "-fPIC",
                        os.path.join(ROOT, "scripts", "fp64_probe.cu"), "-o", so], check=True)
        probe = C.CDLL(so)
        probe.fp64_probe_launch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
        blocks, iters = 148 * 8 * 4, 4096
        buf = torch.empty(blocks * 256, dtype=torch.float64, device="cuda")
        fn = lambda: probe.fp64_probe_launch(buf.data_ptr(), blocks, iters, 0.999999, 1e-6, s.cuda_stream)  # noqa: E731
        med, mn = time_events(torch, fn, s, a.reps)
        dfma = blocks * 256 * iters * probe.fp64_probe_chains()
        probe_rate = dfma / (mn * 1e-3)
        emit({"what": "fp64_probe", "dfma": dfma, "median_ms": med, "min_ms": mn, "tdfma_per_s": probe_rate / 1e12,
              "tflops": 2 * probe_rate / 1e12})

    n = 1 << a.n_log2
    g = torch.Generator(device="cuda").manual_seed(3)
    xd = torch.rand(2 * n, dtype=torch.float64, device="cuda", generator=g).mul_(2).sub_(1)
    yd = torch.empty(2 * n, dtype=torch.float64, device="cuda")
    for name, k, real, D, L in SHAPES:
        node = cb.BatchFirNodeF64(taps_for(cb, k, real), decim=D, interp=L)
        n_in = n // L
        n_out = node.out_len(n_in)
        fn = lambda: node.run_dev(xd.data_ptr(), n_in, yd.data_ptr(), n_out, s.cuda_stream)  # noqa: E731
        med, mn = time_events(torch, fn, s, a.reps)
        terms = n_in * k if L > 1 else n_out * k  # products with real samples
        useful = terms * (2 if real else 4)
        emit({"what": "fir_f64", "shape": name, "taps": k, "real": real, "decim": D, "interp": L, "n_in": n_in,
              "n_out": n_out, "median_ms": med, "min_ms": mn, "gsamples_in_per_s": n_in / (med * 1e6),
              "gsamples_out_per_s": n_out / (med * 1e6), "useful_tdfma_per_s": useful / (med * 1e9) / 1e3,
              "fraction_of_probe": useful / (med * 1e-3) / probe_rate,
              "hbm_gb_per_s": 16 * (n_in + n_out) / (med * 1e6)})
        node.close()
    del xd, yd

    # the price of f64: the f32 filter on the 64-complex-tap shape
    x32 = torch.rand(2 * n, dtype=torch.float32, device="cuda", generator=g).mul_(2).sub_(1)
    y32 = torch.empty(2 * n, dtype=torch.float32, device="cuda")
    node32 = cb.BatchFirNode(taps_for(cb, 64, False).astype(np.complex64))
    fn = lambda: node32.run_dev(x32.data_ptr(), n, y32.data_ptr(), n, s.cuda_stream)  # noqa: E731
    med, mn = time_events(torch, fn, s, a.reps)
    emit({"what": "fir_f32_same_shape", "shape": "64 complex", "n_in": n, "median_ms": med, "min_ms": mn,
          "gsamples_per_s": n / (med * 1e6)})

    # one CPU thread of the reference arithmetic, for context
    rng = np.random.default_rng(0)
    m = 1 << 20
    xc = rng.uniform(-1, 1, m) + 1j * rng.uniform(-1, 1, m)
    t = taps_for(cb, 64, False)
    oracle.build()
    oracle.batch_fir(xc[:4096], t, np.zeros(64, np.complex128))
    t0 = time.perf_counter()
    oracle.batch_fir(xc, t, np.zeros(64, np.complex128))
    dt = time.perf_counter() - t0
    emit({"what": "oracle_orc_batch_fir_c64", "shape": "64 complex", "n_in": m, "s": dt, "msamples_per_s": m / dt / 1e6})

    if a.out:
        with open(a.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
