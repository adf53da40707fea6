#!/usr/bin/env python
"""bench.py -- throughput of the comms-rs FIR / mixer / FFT hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload fir64] [--impl b200|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  The
default workload is BASELINE.json configs[1]: one 64-tap complex-f32 FIR
(BatchFirNode, src/filter/fir_node.rs:146-221) over a 2^28-sample stream.
One JSON line is printed by rank 0:
  value     device-resident throughput (inputs already in HBM), CUDA events, max over ranks
  e2e       same metric through the host-pointer C-ABI call (cb_fir_run ...): pinned
            host buffers, H2D + kernel + D2H inside the timed region
  roofline  algorithmic bytes per launch / mean launch time vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle port of the reference algorithm on one host core (N=1, rank 0)
`--impl reference` times the reference's CPU algorithm (oracle port; the Rust
reference cannot be built in this image) on all host cores instead.
N > 1: one process per GPU (torchrun); each rank owns one overlap-save segment of
the stream (its halo is the K samples before it), no data-path collective ->
weak scaling.
--dump-outputs DIR: the inputs are a seeded counter-based stream, so two builds run with the same arguments can be
compared output for output (see dump_output).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "FIR/FFT Msamples/s"
UNIT = "Msamples/s"
SEED = 20260101
DUMP_BYTES = 64_000_000  # --dump-outputs: all files of one run together, .npy headers included

WORKLOADS = {
    # name: (kind, samples per step per GPU, algorithmic bytes per input sample, description)
    "fir64": ("fir", 1 << 28, 16.0, "64-tap complex-f32 FIR (complex taps) on one 2^28-sample stream per GPU"),
    "fir64_real": ("fir", 1 << 28, 16.0, "64-tap complex-f32 FIR (real-valued rrc taps) on one 2^28-sample stream per GPU"),
    "fir64_iq16": ("fir16", 1 << 28, 8.0, "64-tap complex FIR with i16 IQ on both edges (IQBatchInput -> filter -> IQBatchOutput, src/io/raw_iq.rs): "
                   "4 B in + 4 B out per sample; cast and quantiser run as separate kernels around the f32 filter, so the device-resident "
                   "figure is low against an 8 B/sample roof -- the point of the entry is the PCIe-bound host call"),
    "fir1024": ("fir", 1 << 28, 16.0, "1024-tap complex-f32 FIR (overlap-save fast convolution) on one 2^28-sample stream per GPU"),
    "fir63d5": ("firdec", 1 << 28, 9.6, "63-tap real-valued FIR + DecimateNode(5) (fm_radio.rs filt1 -> dec1) fused, one 2^28-sample stream per GPU"),
    "fir63d5_real": ("firreal", 1 << 28, 4.8, "fm_radio second stage (fm_radio.rs:98-164): real f32 samples -> Complex(x,0) -> 63-tap FIR -> .re -> "
                     "DecimateNode(5), fused, one 2^28-sample real stream per GPU"),
    "fm_radio": ("graph", 1 << 28, 2.16, "examples/fm_radio.rs end to end, one stream per GPU: u8 IQ -> ConvertNode -> filt1 (63 taps) -> /5 -> "
                 "FMDemodNode -> Convert2Node -> filt2 (63 taps) -> Convert3Node -> /5 -> f32 audio; two kernels "
                 "(fused byte front end, fused real second stage), 2^28 IQ samples per step"),
    "fft4096_iq16": ("fft16", 1 << 28, 12.0, "batched 4096-point FFT of i16 IQ samples (IQBatchInput -> FFT, src/io/raw_iq.rs:78-140; the cast is "
                     "folded into the transform's first loads): 4 B in + 8 B out per sample, 2^28 samples per GPU"),
    "fft16": ("fft", 1 << 28, 16.0, "batched 16-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft32": ("fft", 1 << 28, 16.0, "batched 32-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft64": ("fft", 1 << 28, 16.0, "batched 64-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft128": ("fft", 1 << 28, 16.0, "batched 128-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft256": ("fft", 1 << 28, 16.0, "batched 256-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft1024": ("fft", 1 << 28, 16.0, "batched 1024-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft2048": ("fft", 1 << 28, 16.0, "batched 2048-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft16384": ("fft", 1 << 28, 16.0, "batched 16384-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft8192": ("fft", 1 << 28, 16.0, "batched 8192-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft4096": ("fft", 1 << 28, 16.0, "batched 4096-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft65536": ("fft", 1 << 28, 16.0, "batched 65536-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft32768": ("fft", 1 << 28, 16.0, "batched 32768-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft131072": ("fft", 1 << 28, 16.0, "batched 131072-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft524288": ("fft", 1 << 28, 16.0, "batched 524288-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft262144": ("fft", 1 << 28, 16.0, "batched 262144-point FFT over 2^28 complex-f32 samples per GPU"),
    "fft1048576": ("fft", 1 << 28, 16.0, "batched 1048576-point FFT over 2^28 complex-f32 samples per GPU"),
    "freqest": ("est", 1 << 27, 16.0, "frequency_offset_estimate (frequency_estimator.rs:27-42) over 2^27 complex-f64 samples per GPU"),
    "timing10x5": ("est", 1 << 27, 16.0, "TimingEstimator(n=10, d=5, alpha=0.5).push (timing_estimator.rs:85-112, 101-tap f64 filter) "
                   "over 2^27 complex-f64 samples per GPU"),
    "fft1000": ("fft", (1 << 28) // 1000 * 1000, 16.0, "batched 1000-point FFT (chirp-z) over ~2^28 complex-f32 samples per GPU"),
    "fft48000": ("fft", (1 << 28) // 48000 * 48000, 16.0, "batched 48000-point FFT (chirp-z) over ~2^28 complex-f32 samples per GPU"),
    "ifft4096": ("fft", 1 << 28, 16.0, "batched 4096-point IFFT over 2^28 complex-f32 samples per GPU"),
    "mixer": ("mixer", 1 << 28, 16.0, "MixerNode (src/mixer.rs:73-84): y = x e^{j phi}, f64 phase, over 2^28 complex-f32 samples per GPU"),
    "fm": ("fm", 1 << 28, 12.0, "FMDemodNode (src/modulation/analog.rs:22-34) over 2^28 complex-f32 samples per GPU"),
    "chain": ("chain", 1024 * 131072, 8.4, "fm_radio chain x1024 channels per GPU: mixer -> 63-tap FIR -> /10 -> FM demod, "
              "131072-sample batches"),
    "chain5": ("chain", 1024 * 131072, 8.8, "fm_radio as shipped x1024 channels per GPU: 63-tap FIR -> /5 -> FM demod (no mixer), "
               "131072-sample batches"),
    "chain5_u8": ("chain", 1024 * 131072, 2.8, "fm_radio as shipped from raw RTL-SDR bytes x1024 channels per GPU: u8 IQ -> (x-127.5)/127.5 -> "
                  "63-tap FIR -> /5 -> FM demod, fused, 131072-sample batches"),
    "pulse4": ("interp", 1 << 26, 40.0, "BPSK pulse shaping: x4 polyphase 32-tap RRC over 2^26 symbols per GPU (unit = symbols)"),
    "pulse4_b4096": ("interp", 1 << 20, 40.0, "BASELINE configs[0] as specified (examples/single_thread_bpsk.rs:19,39): 2^20 BPSK symbols in 256 "
                     "messages of 4096, x4 / 32-tap RRC pulse shaping, state carried across messages; one step = 256 "
                     "cb_fir_run_dev calls (launch-latency regime; unit = symbols)"),
    "pulse4_i16": ("interp", 1 << 26, 24.0, "BPSK pulse shaping with the example's i16 quantiser fused: x4 polyphase 32-tap RRC -> (8192 x) as i16 "
                   "IQ over 2^26 symbols per GPU (unit = symbols)"),
    "poly8x1024c": ("interp", 1 << 26, 72.0, "x8 polyphase with a fully complex 1024-tap bank (tcgen05, 54 MMAs per tile) over 2^26 symbols "
                    "per GPU (unit = symbols)"),
    "poly8x1024": ("interp", 1 << 27, 72.0, "QPSK symbols -> x8 polyphase, 1024-tap RRC bank (tcgen05 Toeplitz GEMM) over 2^27 symbols per GPU "
                   "= one of the 8 segments of the 2^30-symbol stream, each rank seeded with its 127-symbol halo (unit = symbols)"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="fir64", choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--also", default=None,
                    help="comma-separated extra workloads reported under 'also' on the same line; default: the other BASELINE "
                         "configs when --workload is the default, none otherwise; 'none' disables")
    ap.add_argument("--no-gather", dest="gather", action="store_false",
                    help="N > 1: skip the ordered gather of the output segments (timed apart from the kernels)")
    ap.add_argument("--pageable", action="store_true", help="also time the host-pointer call with pageable host buffers")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each measured workload computed to DIR/<workload>.npy "
                         "(float32 / float64, at most 64 MB in all: larger outputs are sampled at fixed positions)")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs is not None and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if a.also is None:
        a.also = list(ALSO_DEFAULT) if a.workload == "fir64" and a.impl == "b200" else []
    elif a.also.strip().lower() in ("", "none"):
        a.also = []
    else:
        a.also = [w.strip() for w in a.also.split(",") if w.strip()]
        for w in a.also:
            if w not in WORKLOADS:
                ap.error(f"unknown workload in --also: {w}")
    a.dump_bytes = DUMP_BYTES // (1 + len([w for w in a.also if w != a.workload]))
    return a


# ---------------------------------------------------------------------------- workload parameters
def fm_radio_lowpass(n=63):
    k = np.arange(n) - (n - 1) / 2
    return (np.sinc(k / 5) * np.hamming(n) / 5).astype(np.float32).astype(np.complex64)


def rrc_taps(n, sps, beta, cpu=False):
    """rrc_taps (src/util/math.rs:221-280).  GPU arm: the product's host entry (cb_rrc_taps).  CPU legs
    (cpu_baseline, --impl reference): the oracle's restatement, so that the reference arm never maps the product."""
    if cpu:
        import oracle

        return oracle.rrc_taps(n, sps, beta)
    import comms_rs_b200 as cb

    return cb.rrc_taps(n, sps, beta)


def fir_taps(workload, cpu=False):
    nt = 1024 if workload == "fir1024" else 64
    t = rrc_taps(nt, 4.0, 0.25, cpu)
    if workload in ("fir64", "fir1024"):
        t = (t * np.exp(0.1j * np.arange(nt))).astype(np.complex64)
    return t


# ---------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        self.samples, self._stop, self.ok = [], threading.Event(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [v for v in vis.split(",") if v.strip().isdigit()]
            phys = int(ids[index]) if index < len(ids) else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                try:
                    rs = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    rs = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok:
            self.t.join(timeout=2)

    def summary(self, t0, t1):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvml unavailable: " + getattr(self, "err", "")}
        win = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        mhz = sorted(s[1] for s in win)
        bits = 0
        for s in win:
            bits |= s[2]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(v for k, v in self.REASONS.items() if bits & k), "samples": len(win)}


# ---------------------------------------------------------------------------- CPU legs (oracle port)
def cpu_rate(workload, samples, threads):
    """Times the oracle's restatement of the reference algorithm on `samples` units split over
    `threads` independent segments (each seeded with its halo).  Returns (Msamples/s, seconds)."""
    import oracle

    oracle.build()
    kind = WORKLOADS[workload][0]
    per = max(samples // threads, 1)
    if kind == "fft":
        n = int(workload.replace("ifft", "").replace("fft", ""))
        per = max(per // n, 1) * n
    if kind == "fft16":
        per = max(per // 4096, 1) * 4096
    jobs = []
    for i in range(threads):
        x = oracle.synth_uniform_c32(SEED, i * per, per)
        if kind == "fir16":
            t = fir_taps("fir64", cpu=True)
            iq = (x.view(np.float32) * np.float32(32767.0)).astype(np.int16)
            jobs.append(lambda iq=iq, t=t: oracle.quantize_i16(oracle.batch_fir(
                (iq.astype(np.float32) * np.float32(1.0 / 32767.0)).view(np.complex64), t, np.zeros(len(t), np.complex64),
                literal=True, native=True)[0], 8192.0))
        elif kind == "fir":
            t = fir_taps(workload, cpu=True)
            # reference form: per-sample rotate + ordered MACs (src/filter/fir.rs:87-102), release flags
            jobs.append(lambda x=x, t=t: oracle.batch_fir(x, t, np.zeros(len(t), np.complex64), literal=True, native=True))
        elif kind == "fft":
            jobs.append(lambda x=x: oracle.fft(x, n, workload.startswith("ifft")))
        elif kind == "fft16":
            iq = (x.view(np.float32) * np.float32(32767.0)).astype(np.int16)
            jobs.append(lambda iq=iq: oracle.fft((iq.astype(np.float32) * np.float32(1.0 / 32767.0)).view(np.complex64), 4096, False))
        elif kind == "firdec":
            t = fm_radio_lowpass()
            jobs.append(lambda x=x, t=t: oracle.decimate(oracle.batch_fir(x, t, np.zeros(63, np.complex64), literal=True, native=True)[0], 5))
        elif kind == "firreal":
            t = fm_radio_lowpass()
            xr = x.view(np.float32)[:per].astype(np.complex64)  # Convert2Node
            jobs.append(lambda xr=xr, t=t: oracle.decimate(
                oracle.batch_fir(xr, t, np.zeros(63, np.complex64), literal=True, native=True)[0].real.copy(), 5))
        elif kind == "graph":
            t = fm_radio_lowpass()
            b8 = np.clip(x.view(np.float32) * 127.5 + 127.5, 0, 255).astype(np.uint8)

            def whole(b8=b8, t=t):
                z = oracle.u8_to_f32(b8).view(np.complex64)                                  # ConvertNode
                fm = oracle.FmChain(0.0, 0.0, t, 5, do_mix=False, do_fm=True, native=True).run(z)  # filt1, dec1, fm
                f2 = oracle.batch_fir(fm.astype(np.complex64), t, np.zeros(63, np.complex64), literal=True, native=True)[0]
                return oracle.decimate(f2.real.copy(), 5)                                   # Convert3Node, dec2
            jobs.append(whole)
        elif kind == "est":
            x = x.astype(np.complex128)
            if workload == "freqest":
                jobs.append(lambda x=x: oracle.frequency_offset_estimate(x))
            else:
                jobs.append(lambda x=x: oracle.TimingEstimator(10, 5, 0.5).push(x))
        elif kind == "mixer":
            jobs.append(lambda x=x: oracle.Mixer(0.2, 0.123).mix(x))
        elif kind == "fm":
            jobs.append(lambda x=x: oracle.FM().demod(x))
        elif kind == "chain":
            if workload.startswith("chain5"):
                ch = oracle.FmChain(0.0, 0.0, fm_radio_lowpass(), 5, do_mix=False, native=True)
            else:
                ch = oracle.FmChain(-0.7, 0.0, fm_radio_lowpass(), 10, native=True)
            jobs.append(lambda x=x, ch=ch: [ch.run(x[j:j + 131072]) for j in range(0, len(x), 131072)])
        else:
            L, nt = (4, 32) if workload.startswith("pulse4") else (8, 1024)
            if workload == "poly8x1024":
                x = (np.where(x.real >= 0, 1.0, -1.0) + 1j * np.where(x.imag >= 0, 1.0, -1.0)).astype(np.complex64)
            t = rrc_taps(nt, float(L), 0.25, cpu=True)
            st = np.zeros(nt, np.complex64)
            jobs.append(lambda x=x, t=t, st=st: oracle.batch_fir(oracle.upsample(x, L), t, st, literal=True, native=True))
    ths = [threading.Thread(target=j) for j in jobs]
    t0 = time.perf_counter()
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    dt = time.perf_counter() - t0
    return per * threads / dt / 1e6, dt, per * threads


def run_reference(args, rank):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    kind, _, _, desc = WORKLOADS[args.workload]
    rate1 = {"fir16": 8e6, "fft16": 30e6, "fir": 8e6, "fft": 30e6, "chain": 20e6, "interp": 2e6, "mixer": 30e6, "fm": 60e6, "firdec": 8e6, "est": 3e6, "firreal": 8e6, "graph": 8e6}[kind]
    if args.workload.startswith("poly8x1024"):
        rate1 = 1e4
    per_thread = int(min(max(150.0 * rate1 / (args.steps + args.warmup), 1 << 12), 1 << 23))
    sample = per_thread * threads
    for _ in range(args.warmup):
        cpu_rate(args.workload, sample, threads)
    tot_t, tot_n = 0.0, 0
    for _ in range(args.steps):
        _, dt, n = cpu_rate(args.workload, sample, threads)
        tot_t += dt
        tot_n += n
    v = tot_n / tot_t / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64" if kind == "est" else "f32", "data": "synthetic",
        "config": {"workload": args.workload, "description": desc,
                   "note": "reference CPU algorithm (oracle port of the Rust code; no rustc in this image), "
                           "independent segments with halo state, one per host thread"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} units per step ({per_thread} per thread), {args.steps} steps"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------- GPU leg
class Job:
    """One workload bound to one GPU: device buffers, handles, and the per-step launch."""

    def __init__(self, cb, torch, workload, rank):
        self.cb, self.torch, self.workload = cb, torch, workload
        self.kind, self.n, self.bytes_per_unit, self.desc = WORKLOADS[workload]
        # a real (non-NULL) stream: NULL would mean "the handle's own stream" to *_run_dev,
        # and the CUDA events below must sit on the stream the kernels are launched on
        self.tstream = torch.cuda.Stream()
        self.stream = self.tstream.cuda_stream
        assert self.stream != 0
        n = self.n
        self.first = rank * n  # this rank's segment of the global synthetic stream
        self.x = torch.empty(n, dtype=torch.complex64, device="cuda")
        cb.synth_uniform_dev(SEED, self.first, n, self.x.data_ptr(), self.stream)
        self.kernels_per_step = 1
        if self.kind == "fir":
            self.taps = fir_taps(workload)
            self.halo = self._halo(len(self.taps))
            self.node = cb.BatchFirNode(self.taps, self.halo)
            self.y = torch.empty(n, dtype=torch.complex64, device="cuda")
            self.out_bytes = 8 * n
            self.step = lambda: self.node.run_dev(self.x.data_ptr(), n, self.y.data_ptr(), n, self.stream)
            self.step_to = lambda dst: self.node.run_dev(self.x.data_ptr(), n, dst, n, self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_fir_run(self.node._h, hin, n, hout, n, None)
        elif self.kind == "fir16":
            self.taps = fir_taps("fir64")
            self.node = cb.BatchFirNode(self.taps, None)
            xr = torch.view_as_real(self.x)
            self.x16 = (xr * 32767.0).to(torch.int16).contiguous()  # the same synthetic stream as i16 IQ
            self.x8 = self.x16  # (the e2e leg copies `x8` when present)
            self.y = torch.empty(2 * n, dtype=torch.int16, device="cuda")
            self.in_bytes_override = 4 * n
            self.out_bytes = 4 * n
            self.kernels_per_step = 1  # roofline over the whole step (cast + filter + fix-up + quantiser)
            sc_in, sc_out = 1.0 / 32767.0, 8192.0
            self.step = lambda: self.node.run_dev_iq16(self.x16.data_ptr(), n, sc_in, sc_out, self.y.data_ptr(), n, self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_fir_run_iq16(self.node._h, hin, n, sc_in, sc_out, hout, n, None)
        elif self.kind == "fft16":
            self.node = cb.FFTBatchNode(4096, False)
            xr = torch.view_as_real(self.x)
            self.x16 = (xr * 32767.0).to(torch.int16).contiguous()
            self.x8 = self.x16  # (the e2e leg copies `x8` when present)
            self.y = torch.empty(n, dtype=torch.complex64, device="cuda")
            self.in_bytes_override = 4 * n
            self.out_bytes = 8 * n
            sc_in = 1.0 / 32767.0
            self.step = lambda: self.node.run_dev_iq16(self.x16.data_ptr(), n, sc_in, self.y.data_ptr(), self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_fft_run_iq16(self.node._h, hin, n, sc_in, hout)
        elif self.kind == "firdec":
            self.taps = fm_radio_lowpass()
            self.node = cb.BatchFirNode(self.taps, None, decim=5)
            no = -(-n // 5)
            self.y = torch.empty(no, dtype=torch.complex64, device="cuda")
            self.out_bytes = 8 * no
            self.step = lambda: self.node.run_dev(self.x.data_ptr(), n, self.y.data_ptr(), no, self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_fir_run(self.node._h, hin, n, hout, no, None)
        elif self.kind == "fft":
            N = int(workload.replace("ifft", "").replace("fft", ""))
            self.node = cb.FFTBatchNode(N, workload.startswith("ifft"))
            self.y = torch.empty(n, dtype=torch.complex64, device="cuda")
            self.out_bytes = 8 * n
            self.kernels_per_step = 2 if os.environ.get("COMMS_B200_FFT_PATH") in ("fourstep", "rows2", "twopass") and N > 16384 else 1
            self.step = lambda: self.node.run_dev(self.x.data_ptr(), n, self.y.data_ptr(), self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_fft_run(self.node._h, hin, n, hout)
        elif self.kind == "firreal":
            self.taps = fm_radio_lowpass()
            self.node = cb.BatchFirNode(self.taps, None, decim=5)
            no = -(-n // 5)
            self.y = torch.empty(no, dtype=torch.float32, device="cuda")
            self.in_bytes_override = 4 * n  # the first n floats of the synthetic stream
            self.out_bytes = 4 * no
            self.kernels_per_step = 1  # + the 128-sample history update
            self.step = lambda: self.node.run_dev_real(self.x.data_ptr(), n, self.y.data_ptr(), no, self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_fir_run_real(self.node._h, hin, n, hout, no, None)
        elif self.kind == "graph":
            taps = fm_radio_lowpass()
            self.front = cb.ChainBank(1, taps, 5, dphase=None, with_fm=True)
            self.back = cb.BatchFirNode(taps, None, decim=5)
            n1 = -(-n // 5)
            n2 = -(-n1 // 5)
            self.x8 = (torch.view_as_real(self.x) * 127.5 + 127.5).clamp_(0, 255).to(torch.uint8).contiguous()
            self.mid = torch.empty(n1, dtype=torch.float32, device="cuda")
            self.y = torch.empty(n2, dtype=torch.float32, device="cuda")
            self.in_bytes_override = 2 * n
            self.out_bytes = 4 * n2
            self.kernels_per_step = 1  # roofline over the whole step (two kernels + the 128-sample history update)

            def step():
                self.front.run_dev_u8(self.x8.data_ptr(), n, self.mid.data_ptr(), n1, self.stream)
                self.back.run_dev_real(self.mid.data_ptr(), n1, self.y.data_ptr(), n2, self.stream)
            self.step = step
            # end to end: host bytes in, host audio out, the two GPU nodes chained through device buffers (the DeviceBuf
            # edge of INTEGRATION.md section 3) -- only the graph's outer edges cross PCIe
            self.x8_e2e = torch.empty_like(self.x8)
            self.e2e_api = ("cb_copy_h2d_async -> cb_chain_run_u8_dev -> cb_fir_run_real_dev -> cb_copy_d2h_async on one stream, "
                            "pinned host buffers: nodes chained through device buffers, only the graph's outer edges cross PCIe")

            def host_call(hin, hout):
                lib = cb.load()
                rc = lib.cb_copy_h2d_async(self.x8_e2e.data_ptr(), hin, 2 * n, self.stream)
                if rc:
                    return rc
                self.front.run_dev_u8(self.x8_e2e.data_ptr(), n, self.mid.data_ptr(), n1, self.stream)
                self.back.run_dev_real(self.mid.data_ptr(), n1, self.y.data_ptr(), n2, self.stream)
                rc = lib.cb_copy_d2h_async(hout, self.y.data_ptr(), 4 * n2, self.stream)
                self.tstream.synchronize()
                return rc
            self.host_call = host_call
        elif self.kind == "est":
            import ctypes as C
            self.x = self.x.to(torch.complex128)  # the same synthetic stream, widened once outside the timed region
            self.in_bytes_override = 16 * n
            self.out_bytes = 8
            self.kernels_per_step = 1  # + one single-CTA kernel that adds the per-CTA partial sums
            self.result = C.c_double(0.0)
            if workload == "freqest":
                self.step = lambda: cb._lib.check(cb.load().cb_freq_estimate_dev(self.x.data_ptr(), n, C.byref(self.result), self.stream))
                self.host_call = lambda hin, hout: cb.load().cb_freq_estimate(hin, n, C.cast(hout, C.POINTER(C.c_double)))
            else:
                self.node = cb.TimingEstimator(10, 5, 0.5)
                self.step = lambda: cb._lib.check(cb.load().cb_timing_push_dev(self.node._h, self.x.data_ptr(), n, C.byref(self.result), self.stream))
                self.host_call = lambda hin, hout: cb.load().cb_timing_push(self.node._h, hin, n, C.cast(hout, C.POINTER(C.c_double)))
        elif self.kind == "mixer":
            self.node = cb.MixerNode(0.123, 0.2)
            self.y = torch.empty(n, dtype=torch.complex64, device="cuda")
            self.out_bytes = 8 * n
            self.step = lambda: cb._lib.check(cb.load().cb_mixer_run_dev(self.node._h, self.x.data_ptr(), n, self.y.data_ptr(), self.stream))
            self.host_call = lambda hin, hout: cb.load().cb_mixer_run(self.node._h, hin, n, hout)
        elif self.kind == "fm":
            self.node = cb.FMDemodNode()
            self.y = torch.empty(n, dtype=torch.float32, device="cuda")
            self.out_bytes = 4 * n
            self.step = lambda: cb._lib.check(cb.load().cb_fm_run_dev(self.node._h, self.x.data_ptr(), n, self.y.data_ptr(), self.stream))
            self.host_call = lambda hin, hout: cb.load().cb_fm_run(self.node._h, hin, n, hout)
        elif self.kind == "chain":
            C, nb = 1024, 131072
            fc = (np.arange(C) / C - 0.5) * 0.8
            if workload in ("chain5", "chain5_u8"):
                self.node = cb.ChainBank(C, fm_radio_lowpass(), 5, dphase=None, with_fm=True)
            else:
                self.node = cb.ChainBank(C, fm_radio_lowpass(), 10, dphase=-2 * np.pi * fc, with_fm=True)
            no = self.node.out_len(nb)
            self.y = torch.empty(C * no, dtype=torch.float32, device="cuda")
            self.out_bytes = 4 * C * no
            self.step = lambda: self.node.run_dev(self.x.data_ptr(), nb, self.y.data_ptr(), no, self.stream)
            self.host_call = lambda hin, hout: cb.load().cb_chain_run(self.node._h, hin, nb, hout, no, None)
            if workload == "chain5_u8":  # the same synthetic stream, quantised to RTL-SDR bytes once, outside the timed region
                self.x8 = (torch.view_as_real(self.x) * 127.5 + 127.5).clamp_(0, 255).to(torch.uint8).contiguous()
                self.in_bytes_override = 2 * n
                self.step = lambda: self.node.run_dev_u8(self.x8.data_ptr(), nb, self.y.data_ptr(), no, self.stream)
                self.host_call = lambda hin, hout: cb.load().cb_chain_run_u8(self.node._h, hin, nb, hout, no, None)
        else:
            L, nt = (4, 32) if workload.startswith("pulse4") else (8, 1024)
            self.taps = rrc_taps(nt, float(L), 0.25)
            if workload == "poly8x1024c":
                self.taps = (self.taps * np.exp(0.01j * np.arange(nt))).astype(np.complex64)
            if workload == "poly8x1024":  # QPSK symbols (+-1 +- 1j): the sign bits of the counter-hash stream
                torch.cuda.current_stream().wait_stream(self.tstream)
                xr = torch.view_as_real(self.x)
                xr.copy_(torch.where(xr >= 0, 1.0, -1.0))
                torch.cuda.synchronize()
            # this rank's segment of the symbol stream: the nt/L - 1 symbols before it are the reference `state`
            # (zero-stuffed domain, src/filter/fir_node.rs:193-200)
            self.halo = self._halo(nt // L, interp=L, nstate=nt, qpsk=workload == "poly8x1024")
            self.node = cb.BatchFirNode(self.taps, self.halo, interp=L)
            if workload == "pulse4_b4096":
                nb = 4096
                self.messages_per_step = n // nb
                self.y = torch.empty(n * L, dtype=torch.complex64, device="cuda")
                self.out_bytes = 8 * n * L
                xp, yp = self.x.data_ptr(), self.y.data_ptr()

                def step():
                    for m in range(n // nb):
                        self.node.run_dev(xp + 8 * m * nb, nb, yp + 8 * m * nb * L, nb * L, self.stream)
                self.step = step
                self.kernels_per_step = n // nb
                self.e2e_api = "256 host-pointer cb_fir_run calls per step, one per 4096-symbol message (Vec in, Vec out)"

                def host_call(hin, hout):
                    lib = cb.load()
                    for m in range(n // nb):
                        rc = lib.cb_fir_run(self.node._h, hin + 8 * m * nb, nb, hout + 8 * m * nb * L, nb * L, None)
                        if rc:
                            return rc
                    return 0
                self.host_call = host_call
            elif workload == "pulse4_i16":
                self.y = torch.empty(2 * n * L, dtype=torch.int16, device="cuda")
                self.out_bytes = 4 * n * L
                self.step = lambda: self.node.run_dev_i16(self.x.data_ptr(), n, 8192.0, self.y.data_ptr(), n * L, self.stream)
                self.host_call = lambda hin, hout: cb.load().cb_fir_run_i16(self.node._h, hin, n, 8192.0, hout, n * L, None)
            else:
                self.y = torch.empty(n * L, dtype=torch.complex64, device="cuda")
                self.out_bytes = 8 * n * L
                self.step = lambda: self.node.run_dev(self.x.data_ptr(), n, self.y.data_ptr(), n * L, self.stream)
                self.step_to = lambda dst: self.node.run_dev(self.x.data_ptr(), n, dst, n * L, self.stream)
                self.host_call = lambda hin, hout: cb.load().cb_fir_run(self.node._h, hin, n, hout, n * L, None)
        self.in_bytes = getattr(self, "in_bytes_override", 8 * n)

    def _halo(self, k, interp=1, nstate=None, qpsk=False):
        """The k samples before this rank's segment as the reference `state` (newest first; zero-stuffed domain when
        interp > 1; src/filter/fir_node.rs:193-200): what makes segment + halo partitioning exact."""
        if self.first == 0:
            return None
        from comms_rs_b200 import sharding
        t = self.torch.empty(k, dtype=self.torch.complex64, device="cuda")
        self.cb.synth_uniform_dev(SEED, self.first - k, k, t.data_ptr(), self.stream)
        self.torch.cuda.synchronize()
        prev = t.cpu().numpy()
        if qpsk:
            prev = (np.where(prev.real >= 0, 1.0, -1.0) + 1j * np.where(prev.imag >= 0, 1.0, -1.0)).astype(np.complex64)
        return sharding.halo_state(prev, nstate if nstate is not None else k, interp)


def sample_rows(rows, max_rows):
    """Row indices --dump-outputs keeps of an output of `rows` rows: None (all) when they fit, else one row from each
    of `max_rows` equal strata at an offset drawn from SEED -- the same positions on every run and every build."""
    if rows <= max_rows:
        return None
    stride = rows // max_rows
    return np.arange(max_rows, dtype=np.int64) * stride + np.random.default_rng(SEED).integers(0, stride, max_rows)


def dump_output(job, torch, path, max_bytes):
    """Writes the array a caller of the timed path receives from its last step: float32 (complex samples and i16 IQ as
    (re, im) rows) or float64 (the estimators' result), sampled by sample_rows to at most `max_bytes`."""
    torch.cuda.synchronize()
    if job.kind == "est":
        np.save(path, np.array([job.result.value], dtype=np.float64))
        return
    y = job.y
    if y.is_complex():
        y = torch.view_as_real(y)
    elif y.dtype == torch.int16:
        y = y.view(-1, 2)
    idx = sample_rows(y.shape[0], max((max_bytes - 4096) // (4 * y[0].numel()), 1))  # 4 KB: room for the .npy header
    if idx is not None:
        y = y.index_select(0, torch.from_numpy(idx).to(y.device))
    np.save(path, y.float().cpu().numpy())


ALSO_DEFAULT = ["fft1024", "fft4096", "ifft4096", "fft65536", "chain", "pulse4_b4096", "poly8x1024", "fir64_iq16"]
NVLINK_GBS_PER_DIR = 900.0  # NVLink 5, per GPU and direction (B200_PROFILING.md)


class PinnedPair:
    """One pinned input / output buffer pair, grown on demand and shared by all workloads of a run."""

    def __init__(self, cb):
        self.cb, self.h = cb, [None, None]
        self.cap = [0, 0]

    def get(self, in_bytes, out_bytes):
        import ctypes as C
        lib = self.cb.load()
        for i, need in enumerate((in_bytes, out_bytes)):
            if need > self.cap[i]:
                if self.h[i] is not None:
                    lib.cb_buf_release(self.h[i])
                self.h[i] = C.c_void_p()
                self.cb._lib.check(lib.cb_buf_alloc_pinned(need, C.byref(self.h[i])))
                self.cap[i] = need
        return lib.cb_buf_ptr(self.h[0]), lib.cb_buf_ptr(self.h[1])

    def close(self):
        for h in self.h:
            if h is not None:
                self.cb.load().cb_buf_release(h)
        self.h = [None, None]
        self.cap = [0, 0]


def gather_leg(cb, torch, dist, job, rank, world, reps=3):
    """The one collective of the design, timed apart from the kernels: every rank's output segment back into ONE ordered
    stream on rank 0.  (i) cb_gather_segments_to_root_dev (grouped ncclSend/ncclRecv) after the kernels; (ii) the gather
    fused into the producing kernel: rank 0 exports the stream buffer (CUDA IPC), every rank's kernel stores its segment
    straight into it over NVLink.  CUDA events on the launch stream, max over ranks."""
    import ctypes as C

    from comms_rs_b200 import sharding
    lib = cb.load()
    seg_bytes = job.out_bytes
    counts = [seg_bytes] * world
    ids = [sharding.SegmentGather.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    g = sharding.SegmentGather(world, rank, ids[0])
    root = C.c_void_p()
    base = 0
    if rank == 0:
        cb._lib.check(lib.cb_buf_alloc_device(seg_bytes * world, C.byref(root)))
        base = lib.cb_buf_ptr(root)

    def timed(fn, n):
        fn()  # warm-up (NCCL connection set-up, peer mapping faults)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(job.tstream)
        for _ in range(n):
            fn()
        e1.record(job.tstream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms = timed(lambda: g.gather_to_root_dev(job.y.data_ptr(), counts, 1, 0, base, job.stream), reps)
    remote = seg_bytes * (world - 1)
    out = {"algorithm": "gather-to-root: one grouped ncclSend/ncclRecv (cb_gather_segments_to_root_dev), after the kernels",
           "ms": ms, "bytes_into_root": remote, "root_ingress_GBps": remote / (ms * 1e-3) / 1e9,
           "nvlink_GBps_per_dir": NVLINK_GBS_PER_DIR, "frac_of_nvlink": remote / (ms * 1e-3) / 1e9 / NVLINK_GBS_PER_DIR,
           "segments": world, "segment_bytes": seg_bytes}
    # fused: d_out = the root's buffer (peer-mapped) + this rank's offset
    hnd, err = [None], ""
    if rank == 0:
        try:
            hnd[0] = sharding.peer_export(base)
        except Exception as e:  # noqa: BLE001
            err = repr(e)[:200]
    dist.broadcast_object_list(hnd, src=0)
    mapped = base
    if rank != 0 and hnd[0] is not None:
        try:
            mapped = sharding.peer_open(hnd[0])
        except Exception as e:  # noqa: BLE001
            err, mapped = repr(e)[:200], 0
    okt = torch.tensor([1 if (hnd[0] is not None and mapped) else 0], dtype=torch.int32, device="cuda")
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    if int(okt.item()) == 1:  # every rank mapped the buffer: all of them run the timed loop
        dst = mapped + rank * seg_bytes
        ms_f = timed(lambda: job.step_to(dst), reps)
        out["fused_store"] = {"algorithm": "kernel stores straight into rank 0's stream buffer (cb_peer_export/open, NVLink P2P); "
                                           "no collective call, no second pass", "ms_per_step": ms_f,
                              "root_ingress_GBps": remote / (ms_f * 1e-3) / 1e9,
                              "vs_kernel_then_gather_ms": None}
    else:
        out["fused_store"] = {"unavailable": err or "a peer rank could not map the exported buffer"}
    if rank != 0 and mapped:
        try:
            sharding.peer_close(mapped)
        except Exception:  # noqa: BLE001
            pass
    dist.barrier()
    g.close()
    if rank == 0:
        lib.cb_buf_release(root)
    return out


def measure(cb, torch, dist, args, workload, rank, world, local_rank, steps, warmup, pinned, cpu_sample_scale=1.0):
    """One workload on this rank's GPU: device-resident timing, end-to-end timing, roofline, CPU baseline."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    job = Job(cb, torch, workload, rank)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- device-resident: W warm-up steps, then exactly K timed steps
    for _ in range(warmup):
        job.step()
    barrier()
    launches0 = cb.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    t_wall0 = time.perf_counter()
    for i in range(steps):
        ev[i].record(job.tstream)
        job.step()
    ev[steps].record(job.tstream)
    barrier()
    t_wall1 = time.perf_counter()
    launches_dev = cb.launch_count() - launches0
    total_ms = ev[0].elapsed_time(ev[steps])
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    clocks = sampler.summary(t_wall0, t_wall1)
    if args.dump_outputs:  # before the e2e leg, which some workloads run through the same output buffer
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = workload if world == 1 else f"{workload}.rank{rank}"
        dump_output(job, torch, os.path.join(args.dump_outputs, name + ".npy"), args.dump_bytes // world)

    # ---- end to end: host buffers, H2D + kernels + D2H inside the timed region
    e2e = None
    launches_e2e = 0
    if not args.no_e2e:
        lib = cb.load()
        pin, pout = pinned.get(job.in_bytes, job.out_bytes)
        src = job.x8 if hasattr(job, "x8") else job.x
        cb._lib.check(lib.cb_copy_d2h_async(pin, src.data_ptr(), job.in_bytes, job.stream))
        torch.cuda.synchronize()
        k_e2e = max(3, min(steps, 10))

        def time_host(hin, hout, k):
            for _ in range(2):
                cb._lib.check(job.host_call(hin, hout))
            barrier()
            l0 = cb.launch_count()
            t0 = time.perf_counter()
            for _ in range(k):
                cb._lib.check(job.host_call(hin, hout))  # returns when the host output buffer is filled
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return world * job.n * k / float(tt.item()) / 1e6, cb.launch_count() - l0, float(tt.item())

        v, launches_e2e, dt = time_host(pin, pout, k_e2e)
        e2e = {"value": v, "unit": UNIT,
               "h2d_bytes_per_step": job.in_bytes, "d2h_bytes_per_step": job.out_bytes, "steps": k_e2e,
               "h2d_GBps_per_gpu": job.in_bytes * k_e2e / dt / 1e9, "d2h_GBps_per_gpu": job.out_bytes * k_e2e / dt / 1e9,
               "api": getattr(job, "e2e_api", "host-pointer C-ABI call, pinned buffers, 2-lane chunked H2D/kernel/D2H pipeline")}
        if args.pageable and workload == args.workload:
            # what a Rust Vec is: pageable memory on both sides of the same call
            hin = np.empty(job.in_bytes, dtype=np.uint8)
            hout = np.empty(job.out_bytes, dtype=np.uint8)
            import ctypes as C
            C.memmove(hin.ctypes.data, pin, job.in_bytes)
            vp, lp, _ = time_host(hin.ctypes.data, hout.ctypes.data, 3)
            launches_e2e += lp
            e2e["pageable"] = {"value": vp, "unit": UNIT, "steps": 3,
                               "note": "same call with pageable (malloc) host buffers, the memory of a Rust Vec"}
            del hin, hout
    sampler.stop()

    gather = None
    if world > 1 and args.gather and job.kind in ("fir", "interp") and hasattr(job, "step_to"):
        gather = gather_leg(cb, torch, dist, job, rank, world)
        if "fused_store" in gather and "ms_per_step" in gather["fused_store"]:
            gather["fused_store"]["vs_kernel_then_gather_ms"] = total_ms_max / steps + gather["ms"]

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        peak = peaks.get("hbm_gbs")
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        if not peak:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        ms_launch = total_ms / steps / job.kernels_per_step
        alg_bytes = job.bytes_per_unit * job.n / job.kernels_per_step
        achieved = alg_bytes / (ms_launch * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj.get(workload)
            if traffic is not None:
                traffic_src = "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture (" + \
                              tj.get("_sources", {}).get(workload, "see its _comment") + "); not measured in this run"
        except Exception:  # noqa: BLE001
            pass
        line = {
            "metric": METRIC, "value": world * job.n * steps / (total_ms_max * 1e-3) / 1e6, "unit": UNIT,
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": total_ms_max / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64" if job.kind == "est" else "f32", "data": "synthetic",
            "config": {"workload": workload, "description": job.desc, "units_per_step_per_gpu": job.n,
                       "l2": "inputs larger than L2 (%.2f GiB read + %.2f GiB written per step, L2 = 126 MB)"
                             % (job.in_bytes / 2 ** 30, job.out_bytes / 2 ** 30),
                       "parallelism": "one overlap-save segment (or channel/frame block) per GPU with its true halo as the "
                                      "initial state, no data-path collective",
                       "seed": SEED},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": int(launches_dev + launches_e2e),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernels_per_step": job.kernels_per_step,
                         "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": ms_launch},
        }
        if getattr(job, "messages_per_step", 0):
            line["messages"] = {"per_step": job.messages_per_step, "units_per_message": job.n // job.messages_per_step,
                                "us_per_message": 1e3 * total_ms_max / steps / job.messages_per_step,
                                "messages_per_s": job.messages_per_step * steps / (total_ms_max * 1e-3)}
        if gather is not None:
            line["gather"] = gather
        if world == 1 and not args.no_cpu:
            kind = job.kind
            sample = {"fir16": 1 << 26, "fft16": 1 << 27, "fir": 1 << 26, "fft": 1 << 27, "chain": 1 << 26, "interp": 1 << 23, "mixer": 1 << 26, "fm": 1 << 27, "firdec": 1 << 26, "est": 1 << 24, "firreal": 1 << 26, "graph": 1 << 26}[kind]
            if workload == "timing10x5":
                sample = 1 << 22
            if workload.startswith("poly8x1024"):
                sample = 1 << 17
            sample = max(int(sample * cpu_sample_scale), 1 << 12)
            v, dt, n = cpu_rate(workload, sample, 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"first {n} units of the same synthetic stream, {dt:.1f} s, one thread "
                                              "(the reference runs one thread per node)",
                                    "host_cores": os.cpu_count()}
    del job
    torch.cuda.empty_cache()
    return line


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    import comms_rs_b200 as cb

    cb.init(local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pinned = PinnedPair(cb)
    line = measure(cb, torch, dist, args, args.workload, rank, world, local_rank, args.steps, args.warmup, pinned)
    also = {}
    for w in args.also:
        if w == args.workload:
            continue
        sub = measure(cb, torch, dist, args, w, rank, world, local_rank, max(3, min(args.steps, 10)), 3, pinned,
                      cpu_sample_scale=1.0 / 8)
        if rank == 0:
            keep = ("value", "unit", "ms_per_step", "steps", "warmup", "roofline", "e2e", "cpu_baseline", "clocks", "gpu_launches",
                    "messages", "gather", "dtype")
            also[w] = {k: sub[k] for k in keep if k in sub}
            also[w]["description"] = sub["config"]["description"]
            also[w]["units_per_step_per_gpu"] = sub["config"]["units_per_step_per_gpu"]
    pinned.close()
    if rank == 0:
        if also:
            line["also"] = also
            line["gpu_launches"] += sum(v.get("gpu_launches", 0) for v in also.values())
            line["also_note"] = ("the other BASELINE.json configs (plus fir64_iq16: the headline filter with i16 IQ on both edges, "
                                 "src/io/raw_iq.rs, half the PCIe bytes), same protocol as the headline (CUDA events on the launch "
                                 "stream, max over ranks; e2e through the host-pointer C-ABI call; CPU port on one thread on a "
                                 "smaller sample); top-level value / ms_per_step / roofline are the headline workload's alone")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29577", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
