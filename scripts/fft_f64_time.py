"""Time the Complex<f64> FFT (FFTBatchNodeF64.run_dev) with CUDA events on device-resident inputs, against the FP64
FMA rate of scripts/fp64_probe.cu measured in the same process.

    python scripts/fft_f64_time.py [--n-log2 26] [--reps 10] [--out results.jsonl]

Each call transforms 2^n-log2 complex f64 points (2^26: 1 GiB in, 1 GiB out, larger than L2).  Each size is warmed
up, then timed over --reps calls: median and minimum.  Reported per size: Gsamples/s, the fraction of the 6539.9 GB/s
copy roof at 32 B/sample (16 in + 16 out), and the fraction of the probe's FP64 rate taken by the transform's nominal
5 N log2 N flop per frame (counted as FMA-equivalent pairs).  Also timed, for context: the f32 FFTBatchNode at the
same sizes and one CPU thread of scipy.fft on complex128 (2^20 points).  Prints one JSON line per result, the first
with the card's name and power limit.  Writes nothing in the tree; the probe is built in a temporary directory."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [16, 1024, 4096, 8192, 65536, 1 << 20, 1000, 48000, 100]
ROOF_GBS = 6539.9


def time_events(torch, fn, stream, reps, warm=2):
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


def fp64_rate(torch, tmp):
    so = os.path.join(tmp, "fp64_probe.so")
    subprocess.run(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared",
                    "-Xcompiler", "-fPIC", os.path.join(ROOT, "scripts", "fp64_probe.cu"), "-o", so], check=True)
    lib = C.CDLL(so)
    lib.fp64_probe_launch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
    blocks, iters = 148 * 8, 1 << 14
    out = torch.empty(blocks * 256, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream()
    med, _ = time_events(torch, lambda: lib.fp64_probe_launch(out.data_ptr(), blocks, iters, 0.999, 1e-3, st.cuda_stream),
                         st, 5)
    return blocks * 256 * iters * lib.fp64_probe_chains() / (med * 1e-3)  # DFMA/s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-log2", type=int, default=26)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import comms_rs_b200 as cb

    cb.init(0)
    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    emit({"gpu": q, "points_per_call": 1 << args.n_log2, "reps": args.reps})
    with tempfile.TemporaryDirectory() as tmp:
        rate = fp64_rate(torch, tmp)
    emit({"fp64_probe_dfma_per_s": rate})
    total = 1 << args.n_log2
    st = torch.cuda.Stream()  # a stream of its own: a NULL stream would send the work to the handle's stream
    d_in = torch.rand(2 * total, dtype=torch.float64, device="cuda") * 2 - 1
    d_out = torch.empty_like(d_in)
    for n in SIZES:
        m = total // n * n
        node = cb.FFTBatchNodeF64(n)
        med, mn = time_events(torch, lambda: node.run_dev(d_in.data_ptr(), m, d_out.data_ptr(), st.cuda_stream), st,
                              args.reps)
        gsps = m / (med * 1e-3) / 1e9
        flop = 5 * m * math.log2(n) if n > 1 else 0.0
        emit({"what": "fft_f64", "n": n, "path": ["direct", "frames", "two-step", "chirp-z"][_path(n)],
              "ms_median": med, "ms_min": mn, "gsamples_per_s": gsps,
              "frac_copy_roof_32B": gsps * 32 / ROOF_GBS, "frac_fp64_rate": flop / 2 / (med * 1e-3) / rate})
        del node
        x32 = d_in[:2 * m].to(torch.float32)
        o32 = torch.empty_like(x32)
        node32 = cb.FFTBatchNode(n)
        med32, _ = time_events(torch, lambda: node32.run_dev(x32.data_ptr(), m, o32.data_ptr(), st.cuda_stream), st,
                               args.reps)
        emit({"what": "fft_f32", "n": n, "ms_median": med32, "gsamples_per_s": m / (med32 * 1e-3) / 1e9})
        del node32, x32, o32
    import scipy.fft

    xc = np.random.default_rng(0).standard_normal(1 << 21).view(np.complex128)
    for n in SIZES:
        f = xc[: (1 << 20) // n * n].reshape(-1, n)
        t = time.perf_counter()
        scipy.fft.fft(f, axis=1, workers=1)
        dt = time.perf_counter() - t
        emit({"what": "scipy_fft_complex128_1thread", "n": n, "gsamples_per_s": f.size / dt / 1e9})
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("".join(json.dumps(d) + "\n" for d in lines))


def _path(n):
    pow2 = n & (n - 1) == 0
    if pow2 and n >= 8:
        return 1 if n <= 4096 else 2
    return 0 if pow2 or n <= 128 else 3


if __name__ == "__main__":
    main()
