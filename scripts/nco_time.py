"""Time NcoNode.run_dev on 2^28 phase errors with CUDA events (the bench has no NCO workload).

    python scripts/nco_time.py [--n-log2 28] [--reps 20]

Prints one JSON line: the device name and power limit, the median and minimum time per call and the rate in
Msamples/s.  The library is the one of the tree this script sits in."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-log2", type=int, default=28)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    import torch

    import comms_rs_b200 as cb

    cb.init(0)
    n = (1 << a.n_log2) - 1  # at most 2^29 - 1 per call
    g = torch.Generator(device="cuda").manual_seed(1)
    perr = (torch.rand(n, device="cuda", dtype=torch.float64, generator=g) - 0.5) * 1e-3
    out = torch.empty(2 * n, device="cuda", dtype=torch.float64)
    node = cb.NcoNode(0.37, 0.5)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(3):
        node.run_dev(perr.data_ptr(), n, out.data_ptr(), s.cuda_stream)
    s.synchronize()
    times = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        node.run_dev(perr.data_ptr(), n, out.data_ptr(), s.cuda_stream)
        e1.record(s)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    times.sort()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip()
    print(json.dumps({"what": "nco_run_dev", "n": n, "gpu": q, "median_ms": times[len(times) // 2],
                      "min_ms": times[0], "msamples_per_s": n / (times[len(times) // 2] * 1e3)}))


if __name__ == "__main__":
    main()
