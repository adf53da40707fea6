"""Host-side mirror of the comms-rs node structs on the hot path, over the C ABI.

Same names, constructor arguments and `run()` meaning as the reference:
  BatchFirNode / FirNode   src/filter/fir_node.rs:43-221
  PulseNode                src/pulse.rs:36-92
  DecimateNode/UpsampleNode src/util/resample_node.rs:18-131
  MixerNode                src/mixer.rs:91-148
  FFTBatchNode/FFTSampleNode src/fft/fft_node.rs:26-168
  FMDemodNode              src/modulation/analog_node.rs:18-52
`run(host array) -> host array` is the drop-in Vec-in / Vec-out form;
`run_dev(ptr, n, out_ptr, ...)` chains device buffers on a stream.  All
arithmetic happens in libcomms_b200.so; nothing here computes.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import CbError, NodeError, check, node_error

_vp, _sz = C.c_void_p, C.c_size_t


def _c32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.complex64))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_vp)


class _Handle:
    _destroy = None

    def __init__(self):
        self._h = _vp()

    def close(self):
        if getattr(self, "_h", None) is not None and self._h and _lib._LIB is not None:
            getattr(_lib.load(), self._destroy)(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BatchFirNode(_Handle):
    """BatchFirNode::new(taps, state) (src/filter/fir_node.rs:193-211) with the
    neighbouring Upsample/Decimate nodes optionally fused (interp / decim)."""

    _destroy = "cb_fir_destroy"

    def __init__(self, taps, state=None, decim: int = 1, interp: int = 1):
        super().__init__()
        t = _c32(taps)
        s = None if state is None else _c32(state)
        check(_lib.load().cb_fir_create(_ptr(t), len(t), None if s is None else _ptr(s), 0 if s is None else len(s),
                                        decim, interp, C.byref(self._h)))

    def out_len(self, n_in: int) -> int:
        m = _sz()
        check(_lib.load().cb_fir_out_len(self._h, n_in, C.byref(m)))
        return m.value

    def run(self, samples) -> np.ndarray:
        x = _c32(samples)
        out = np.empty(self.out_len(len(x)), dtype=np.complex64)
        m = _sz()
        try:
            check(_lib.load().cb_fir_run(self._h, _ptr(x), len(x), _ptr(out), len(out), C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out[: m.value]

    def run_dev(self, d_in: int, n_in: int, d_out: int, out_cap: int, stream: int = 0) -> int:
        m = _sz()
        check(_lib.load().cb_fir_run_dev(self._h, d_in, n_in, d_out, out_cap, C.byref(m), stream))
        return m.value

    def run_real(self, x) -> np.ndarray:
        """Real samples in, real parts out: Convert2Node -> this filter -> Convert3Node [-> DecimateNode]
        (examples/fm_radio.rs:98-164) in one call."""
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float32))
        n = _sz()
        check(_lib.load().cb_fir_out_len(self._h, len(x), C.byref(n)))
        out = np.empty(n.value, dtype=np.float32)
        m = _sz()
        try:
            check(_lib.load().cb_fir_run_real(self._h, _ptr(x), len(x), _ptr(out), n.value, C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out[: m.value]

    def run_dev_real(self, d_in: int, n_in: int, d_out: int, out_cap: int, stream: int = 0) -> int:
        """Same on device buffers: n_in floats in, out_cap floats of room; returns the number of outputs."""
        m = _sz()
        check(_lib.load().cb_fir_run_real_dev(self._h, d_in, n_in, d_out, out_cap, C.byref(m), stream))
        return m.value

    def run_i16(self, x, scale: float = 8192.0) -> np.ndarray:
        """Host Vec in, interleaved i16 IQ out ([n_out, 2] int16): filter + `(scale * x) as i16`."""
        x = _c32(x)
        n = _sz()
        check(_lib.load().cb_fir_out_len(self._h, len(x), C.byref(n)))
        out = np.empty((n.value, 2), dtype=np.int16)
        m = _sz()
        try:
            check(_lib.load().cb_fir_run_i16(self._h, _ptr(x), len(x), float(scale), _ptr(out), n.value, C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out[: m.value]

    def run_dev_i16(self, d_in: int, n_in: int, scale: float, d_out: int, out_cap: int, stream: int = 0) -> int:
        """Filter + `(scale * x) as i16` (examples/single_thread_bpsk.rs:40-48); d_out: 2*out_cap int16."""
        m = _sz()
        check(_lib.load().cb_fir_run_dev_i16(self._h, d_in, n_in, float(scale), d_out, out_cap, C.byref(m), stream))
        return m.value

    def run_iq16(self, iq, in_scale: float = 1.0, out_scale: float = 1.0) -> np.ndarray:
        """i16 IQ in ([n, 2] int16, what IQBatchInput reads: src/io/raw_iq.rs:78-140), i16 IQ out ([n_out, 2]):
        x = in_scale * (i16 as f32) -> this filter -> (out_scale * y) as i16."""
        x = np.ascontiguousarray(np.asarray(iq, dtype=np.int16)).reshape(-1, 2)
        n = _sz()
        check(_lib.load().cb_fir_out_len(self._h, len(x), C.byref(n)))
        out = np.empty((n.value, 2), dtype=np.int16)
        m = _sz()
        try:
            check(_lib.load().cb_fir_run_iq16(self._h, _ptr(x), len(x), float(in_scale), float(out_scale), _ptr(out), n.value, C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out[: m.value]

    def run_dev_iq16(self, d_in: int, n_in: int, in_scale: float, out_scale: float, d_out: int, out_cap: int, stream: int = 0) -> int:
        m = _sz()
        check(_lib.load().cb_fir_run_dev_iq16(self._h, d_in, n_in, float(in_scale), float(out_scale), d_out, out_cap, C.byref(m), stream))
        return m.value

    @property
    def state(self) -> np.ndarray:
        n = _sz()
        check(_lib.load().cb_fir_state_len(self._h, C.byref(n)))
        st = np.empty(n.value, dtype=np.complex64)
        check(_lib.load().cb_fir_get_state(self._h, _ptr(st), n.value))
        return st

    @state.setter
    def state(self, value):
        s = _c32(value)
        check(_lib.load().cb_fir_set_state(self._h, _ptr(s), len(s)))

    @property
    def stream(self) -> int:
        return _lib.load().cb_fir_stream(self._h) or 0


class FirNode(BatchFirNode):
    """FirNode (src/filter/fir_node.rs:43-114): one sample per run()."""

    def run(self, sample) -> np.complex64:  # type: ignore[override]
        return super().run(np.asarray([sample], dtype=np.complex64))[0]


class PulseNode(BatchFirNode):
    """PulseNode::new(taps, sam_per_sym) (src/pulse.rs:71-80): one symbol in,
    `sam_per_sym` samples out; run() also accepts a batch of symbols."""

    def __init__(self, taps, sam_per_sym: int):
        if sam_per_sym < 1:
            raise NodeError(NodeError.DataError, "sam_per_sym must be >= 1")
        super().__init__(taps, None, decim=1, interp=sam_per_sym)
        self.sam_per_sym = sam_per_sym


def _c128(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.complex128))


class BatchFirNodeF64(_Handle):
    """BatchFirNode<Complex<f64>> (src/filter/fir_node.rs:193-211) over complex128, with the neighbouring
    Upsample/Decimate nodes optionally fused (interp / decim).  Every output is the fixed FMA chain stated in
    include/comms_b200.h (cb_fir_f64), so call splits and host/device entries give the same bits."""

    _destroy = "cb_fir_f64_destroy"

    def __init__(self, taps, state=None, decim: int = 1, interp: int = 1):
        super().__init__()
        t = _c128(taps)
        s = None if state is None else _c128(state)
        check(_lib.load().cb_fir_f64_create(_ptr(t), len(t), None if s is None else _ptr(s), 0 if s is None else len(s),
                                            decim, interp, C.byref(self._h)))

    def out_len(self, n_in: int) -> int:
        m = _sz()
        check(_lib.load().cb_fir_f64_out_len(self._h, n_in, C.byref(m)))
        return m.value

    def run(self, samples) -> np.ndarray:
        x = _c128(samples)
        out = np.empty(self.out_len(len(x)), dtype=np.complex128)
        m = _sz()
        try:
            check(_lib.load().cb_fir_f64_run(self._h, _ptr(x), len(x), _ptr(out), len(out), C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out[: m.value]

    def run_dev(self, d_in: int, n_in: int, d_out: int, out_cap: int, stream: int = 0) -> int:
        """n_in complex f64 in, out_cap of room; device pointers, 16-byte aligned.  Returns the number of outputs."""
        m = _sz()
        check(_lib.load().cb_fir_f64_run_dev(self._h, d_in, n_in, d_out, out_cap, C.byref(m), stream))
        return m.value

    @property
    def state(self) -> np.ndarray:
        n = _sz()
        check(_lib.load().cb_fir_f64_state_len(self._h, C.byref(n)))
        st = np.empty(n.value, dtype=np.complex128)
        check(_lib.load().cb_fir_f64_get_state(self._h, _ptr(st), n.value))
        return st

    @state.setter
    def state(self, value):
        s = _c128(value)
        check(_lib.load().cb_fir_f64_set_state(self._h, _ptr(s), len(s)))

    @property
    def stream(self) -> int:
        return _lib.load().cb_fir_f64_stream(self._h) or 0


class FirNodeF64(BatchFirNodeF64):
    """FirNode<Complex<f64>> (src/filter/fir_node.rs:43-114): one sample per run()."""

    def run(self, sample) -> np.complex128:  # type: ignore[override]
        return super().run(np.asarray([sample], dtype=np.complex128))[0]


class PulseNodeF64(BatchFirNodeF64):
    """PulseNode<f64>::new(taps, sam_per_sym) (src/pulse.rs:71-80): one symbol in, `sam_per_sym` samples out;
    run() also accepts a batch of symbols."""

    def __init__(self, taps, sam_per_sym: int):
        if sam_per_sym < 1:
            raise NodeError(NodeError.DataError, "sam_per_sym must be >= 1")
        super().__init__(taps, None, decim=1, interp=sam_per_sym)
        self.sam_per_sym = sam_per_sym


class _Resample:
    _fn = ""

    def __init__(self, rate: int):
        self.rate = int(rate)

    def _len(self, n: int) -> int:
        raise NotImplementedError

    def run(self, data) -> np.ndarray:
        a = np.ascontiguousarray(data)
        elem = a.dtype.itemsize * int(np.prod(a.shape[1:], dtype=np.int64))
        out = np.empty((self._len(len(a)),) + a.shape[1:], dtype=a.dtype)
        m = _sz()
        try:
            check(getattr(_lib.load(), self._fn)(_ptr(a), len(a), elem, self.rate, _ptr(out), len(out), C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out[: m.value]

    def run_dev(self, d_in: int, n: int, elem_bytes: int, d_out: int, out_cap: int, stream: int = 0) -> int:
        m = _sz()
        check(getattr(_lib.load(), self._fn + "_dev")(d_in, n, elem_bytes, self.rate, d_out, out_cap, C.byref(m), stream))
        return m.value


class DecimateNode(_Resample):
    """DecimateNode::new(dec_rate) (src/util/resample_node.rs:23-31)."""

    _fn = "cb_decimate"

    def _len(self, n):
        return n if self.rate <= 1 else -(-n // self.rate)


class UpsampleNode(_Resample):
    """UpsampleNode::new(ups_rate) (src/util/resample_node.rs:87-95)."""

    _fn = "cb_upsample"

    def _len(self, n):
        return n if self.rate <= 1 else n * self.rate


class MixerNode(_Handle):
    """MixerNode::new(dphase, phase) (src/mixer.rs:128-134) -- note the order."""

    _destroy = "cb_mixer_destroy"

    def __init__(self, dphase: float, phase: float | None = None):
        super().__init__()
        check(_lib.load().cb_mixer_create(float(dphase), 0.0 if phase is None else float(phase), C.byref(self._h)))

    def run(self, samples):
        scalar = np.ndim(samples) == 0
        x = _c32(np.atleast_1d(samples))
        out = np.empty_like(x)
        try:
            check(_lib.load().cb_mixer_run(self._h, _ptr(x), len(x), _ptr(out)))
        except CbError as e:
            raise node_error(e) from e
        return out[0] if scalar else out

    def run_dev(self, d_in: int, n: int, d_out: int, stream: int = 0) -> None:
        check(_lib.load().cb_mixer_run_dev(self._h, d_in, n, d_out, stream))

    @property
    def phase(self) -> float:
        p = C.c_double()
        check(_lib.load().cb_mixer_get_phase(self._h, C.byref(p), None))
        return p.value

    @phase.setter
    def phase(self, v: float):
        check(_lib.load().cb_mixer_set_phase(self._h, float(v)))

    @property
    def dphase(self) -> float:
        d = C.c_double()
        check(_lib.load().cb_mixer_get_phase(self._h, None, C.byref(d)))
        return d.value


class NcoNode(_Handle):
    """NcoNode::new(dphase, phase) (src/demodulation/nco.rs:112-127).  run(perr) takes one phase error (the reference
    contract: f64 in, Complex<f64> out) or a batch of them -- the batching shim that lets a vector of loop-filter
    outputs feed GPU nodes: out[k] = exp(j * phase_k) with Nco::push applied in order (nco.rs:71-77)."""

    _destroy = "cb_nco_destroy"

    def __init__(self, dphase: float, phase: float | None = None):
        super().__init__()
        check(_lib.load().cb_nco_create(float(dphase), 0.0 if phase is None else float(phase), C.byref(self._h)))

    def run(self, perr):
        scalar = np.ndim(perr) == 0
        e = np.ascontiguousarray(np.atleast_1d(np.asarray(perr, dtype=np.float64)))
        out = np.empty(len(e), dtype=np.complex128)
        try:
            check(_lib.load().cb_nco_run(self._h, _ptr(e), len(e), _ptr(out)))
        except CbError as ex:
            raise node_error(ex) from ex
        return out[0] if scalar else out

    def run_dev(self, d_perr: int, n: int, d_out: int, stream: int = 0) -> None:
        """n doubles in, n complex f64 out, device pointers."""
        check(_lib.load().cb_nco_run_dev(self._h, d_perr, n, d_out, stream))

    @property
    def phase(self) -> float:
        p = C.c_double()
        check(_lib.load().cb_nco_get_phase(self._h, C.byref(p), None))
        return p.value

    @phase.setter
    def phase(self, v: float):
        check(_lib.load().cb_nco_set_phase(self._h, float(v)))

    @property
    def dphase(self) -> float:
        d = C.c_double()
        check(_lib.load().cb_nco_get_phase(self._h, None, C.byref(d)))
        return d.value


class FFTBatchNode(_Handle):
    """FFTBatchNode::new(fft_size, ifft) (src/fft/fft_node.rs:65-74).  run() takes
    one frame (the reference contract) or several contiguous frames."""

    _destroy = "cb_fft_destroy"

    def __init__(self, fft_size: int, ifft: bool = False):
        super().__init__()
        self.fft_size = int(fft_size)
        check(_lib.load().cb_fft_create(self.fft_size, int(bool(ifft)), C.byref(self._h)))

    def run(self, data) -> np.ndarray:
        x = _c32(data).reshape(-1)
        out = np.empty_like(x)
        try:
            check(_lib.load().cb_fft_run(self._h, _ptr(x), len(x), _ptr(out)))
        except CbError as e:
            raise node_error(e) from e
        return out

    def run_dev(self, d_in: int, n_in: int, d_out: int, stream: int = 0) -> None:
        check(_lib.load().cb_fft_run_dev(self._h, d_in, n_in, d_out, stream))


def _fft_run_iq16(self, iq, in_scale: float = 1.0) -> np.ndarray:
    """i16 IQ frames in ([n, 2] int16), complex f32 spectra out: x = in_scale * (i16 as f32)."""
    x = np.ascontiguousarray(np.asarray(iq, dtype=np.int16)).reshape(-1, 2)
    out = np.empty(len(x), dtype=np.complex64)
    try:
        check(_lib.load().cb_fft_run_iq16(self._h, _ptr(x), len(x), float(in_scale), _ptr(out)))
    except CbError as e:
        raise node_error(e) from e
    return out


def _fft_run_dev_iq16(self, d_in: int, n_in: int, in_scale: float, d_out: int, stream: int = 0) -> None:
    check(_lib.load().cb_fft_run_dev_iq16(self._h, d_in, n_in, float(in_scale), d_out, stream))


FFTBatchNode.run_iq16 = _fft_run_iq16
FFTBatchNode.run_dev_iq16 = _fft_run_dev_iq16


class FFTSampleNode(FFTBatchNode):
    """FFTSampleNode (src/fft/fft_node.rs:101-168, #[aggregate]): collects
    samples; run() returns None until fft_size samples have arrived."""

    def __init__(self, fft_size: int, ifft: bool = False):
        super().__init__(fft_size, ifft)
        self._acc: list = []

    def run(self, sample):  # type: ignore[override]
        self._acc.append(sample)
        if len(self._acc) == self.fft_size:
            frame, self._acc = self._acc, []
            return super().run(np.asarray(frame, dtype=np.complex64))
        return None


class FFTBatchNodeF64(_Handle):
    """FFTBatchNode<Complex<f64>> (src/fft/fft_node.rs:65-74) over complex128: the transform the reference runs in f64
    (src/fft/mod.rs:73-96), with the per-bin bound, determinism and edges stated in include/comms_b200.h (cb_fft_f64).
    run() takes one frame or several contiguous frames."""

    _destroy = "cb_fft_f64_destroy"

    def __init__(self, fft_size: int, ifft: bool = False):
        super().__init__()
        self.fft_size = int(fft_size)
        check(_lib.load().cb_fft_f64_create(self.fft_size, int(bool(ifft)), C.byref(self._h)))

    def run(self, data) -> np.ndarray:
        x = _c128(data).reshape(-1)
        out = np.empty_like(x)
        try:
            check(_lib.load().cb_fft_f64_run(self._h, _ptr(x), len(x), _ptr(out)))
        except CbError as e:
            raise node_error(e) from e
        return out

    def run_dev(self, d_in: int, n_in: int, d_out: int, stream: int = 0) -> None:
        """n_in complex f64 in and out; device pointers, 16-byte aligned."""
        check(_lib.load().cb_fft_f64_run_dev(self._h, d_in, n_in, d_out, stream))


class FFTSampleNodeF64(FFTBatchNodeF64):
    """FFTSampleNode<Complex<f64>> (src/fft/fft_node.rs:101-168, #[aggregate]): collects samples; run() returns None
    until fft_size samples have arrived."""

    def __init__(self, fft_size: int, ifft: bool = False):
        super().__init__(fft_size, ifft)
        self._acc: list = []

    def run(self, sample):  # type: ignore[override]
        self._acc.append(sample)
        if len(self._acc) == self.fft_size:
            frame, self._acc = self._acc, []
            return super().run(np.asarray(frame, dtype=np.complex128))
        return None


class FMDemodNode(_Handle):
    """FMDemodNode::new() (src/modulation/analog_node.rs:43-52)."""

    _destroy = "cb_fm_destroy"

    def __init__(self):
        super().__init__()
        check(_lib.load().cb_fm_create(C.byref(self._h)))

    def run(self, samples) -> np.ndarray:
        x = _c32(samples)
        out = np.empty(len(x), dtype=np.float32)
        try:
            check(_lib.load().cb_fm_run(self._h, _ptr(x), len(x), _ptr(out)))
        except CbError as e:
            raise node_error(e) from e
        return out

    def run_dev(self, d_in: int, n: int, d_out: int, stream: int = 0) -> None:
        check(_lib.load().cb_fm_run_dev(self._h, d_in, n, d_out, stream))


class ChainBank(_Handle):
    """`channels` independent [MixerNode] -> BatchFirNode -> DecimateNode -> [FMDemodNode]
    chains fused in one kernel (examples/fm_radio.rs:144-164 generalised)."""

    _destroy = "cb_chain_destroy"

    def __init__(self, channels: int, taps, decim: int, dphase=None, phase=None, with_fm: bool = True):
        super().__init__()
        t = _c32(taps)
        d = None if dphase is None else np.ascontiguousarray(np.broadcast_to(np.asarray(dphase, np.float64), (channels,)))
        p = None if phase is None else np.ascontiguousarray(np.broadcast_to(np.asarray(phase, np.float64), (channels,)))
        self.channels, self.with_fm, self.decim = int(channels), bool(with_fm), int(decim)
        check(_lib.load().cb_chain_create(self.channels, None if d is None else _ptr(d), None if p is None else _ptr(p),
                                          _ptr(t), len(t), self.decim, int(self.with_fm), C.byref(self._h)))

    def out_len(self, n_in: int) -> int:
        m = _sz()
        check(_lib.load().cb_chain_out_len(self._h, n_in, C.byref(m)))
        return m.value

    def run(self, x) -> np.ndarray:
        x = _c32(x).reshape(self.channels, -1)
        n_in = x.shape[1]
        no = self.out_len(n_in)
        out = np.empty((self.channels, no), dtype=np.float32 if self.with_fm else np.complex64)
        m = _sz()
        try:
            check(_lib.load().cb_chain_run(self._h, _ptr(x), n_in, _ptr(out), no, C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out

    def run_u8(self, iq) -> np.ndarray:
        """Raw RTL-SDR bytes in ([channels, n_in, 2] uint8: I, Q), ConvertNode (examples/fm_radio.rs:84-87) fused."""
        b = np.ascontiguousarray(np.asarray(iq, dtype=np.uint8)).reshape(self.channels, -1, 2)
        n_in = b.shape[1]
        no = self.out_len(n_in)
        out = np.empty((self.channels, no), dtype=np.float32 if self.with_fm else np.complex64)
        m = _sz()
        try:
            check(_lib.load().cb_chain_run_u8(self._h, _ptr(b), n_in, _ptr(out), no, C.byref(m)))
        except CbError as e:
            raise node_error(e) from e
        return out

    def run_dev_u8(self, d_in: int, n_in: int, d_out: int, out_cap: int, stream: int = 0) -> int:
        m = _sz()
        check(_lib.load().cb_chain_run_u8_dev(self._h, d_in, n_in, d_out, out_cap, C.byref(m), stream))
        return m.value

    def run_dev(self, d_in: int, n_in: int, d_out: int, out_cap: int, stream: int = 0) -> int:
        m = _sz()
        check(_lib.load().cb_chain_run_dev(self._h, d_in, n_in, d_out, out_cap, C.byref(m), stream))
        return m.value


# ------------------------------------------------------------------ edges
def real_to_complex_dev(d_in: int, n: int, d_out: int, stream: int = 0) -> None:
    """Convert2Node of examples/fm_radio.rs:98-118: x -> Complex(x, 0)."""
    check(_lib.load().cb_real_to_complex_dev(d_in, n, d_out, stream))


def complex_real_dev(d_in: int, n: int, d_out: int, stream: int = 0) -> None:
    """Convert3Node of examples/fm_radio.rs:122-142: z -> z.re."""
    check(_lib.load().cb_complex_real_dev(d_in, n, d_out, stream))


def convert_u8_dev(d_in: int, n_samples: int, d_out: int, stream: int = 0) -> None:
    """(u8 I, u8 Q) -> complex f32, (x - 127.5) / 127.5 (examples/fm_radio.rs:84-87)."""
    check(_lib.load().cb_convert_u8_dev(d_in, n_samples, d_out, stream))


def convert_i16_dev(d_in: int, n_samples: int, scale: float, d_out: int, stream: int = 0) -> None:
    """Interleaved i16 IQ (src/io/raw_iq.rs) -> scale * (x as f32)."""
    check(_lib.load().cb_convert_i16_dev(d_in, n_samples, float(scale), d_out, stream))


def rrc_taps(n_taps: int, sam_per_sym: float, beta: float, dtype=np.complex64) -> np.ndarray:
    """rrc_taps::<T> (src/util/math.rs:221-280): root-raised-cosine taps, imaginary parts 0.
    Raises NodeError-style ValueError("InvalidRolloffError") for beta outside [0, 1]."""
    f64 = np.dtype(dtype) == np.complex128
    out = np.empty(n_taps, dtype=np.complex128 if f64 else np.complex64)
    fn = _lib.load().cb_rrc_taps_f64 if f64 else _lib.load().cb_rrc_taps
    try:
        check(fn(int(n_taps), float(sam_per_sym), float(beta), _ptr(out)))
    except CbError as e:
        raise ValueError("InvalidRolloffError") from e
    return out


def qfilt_taps(n_taps: int, alpha: float, sam_per_sym: int) -> np.ndarray:
    """qfilt_taps (src/util/math.rs:307-342): Mengali's q(t), f64; an even n_taps is incremented by one."""
    out = np.empty(n_taps + 1, dtype=np.float64)
    m = C.c_uint32(0)
    try:
        check(_lib.load().cb_qfilt_taps_f64(int(n_taps), float(alpha), int(sam_per_sym), _ptr(out), C.byref(m)))
    except CbError as e:
        raise ValueError("InvalidRolloffError") from e
    return out[:m.value].copy()


def frequency_offset_estimate(samples) -> float:
    """frequency_offset_estimate (src/demodulation/frequency_estimator.rs:27-42): carrier offset in
    radians/sample from complex f64 samples (host array)."""
    x = np.ascontiguousarray(np.asarray(samples, dtype=np.complex128))
    est = C.c_double(0.0)
    check(_lib.load().cb_freq_estimate(_ptr(x), len(x), C.byref(est)))
    return est.value


def frequency_offset_estimate_dev(d_samples: int, n: int, stream: int = 0) -> float:
    """Same on n complex f64 samples already in device memory."""
    est = C.c_double(0.0)
    check(_lib.load().cb_freq_estimate_dev(d_samples, n, C.byref(est), stream))
    return est.value


class TimingEstimator:
    """TimingEstimator (src/demodulation/timing_estimator.rs:13-112): new(n, d, alpha); push(samples) -> estimate
    in samples.  TimingEstimatorNode (timing_estimator.rs:116-137) is the same object: run = push."""

    def __init__(self, n: int, d: int, alpha: float):
        self._h = C.c_void_p()
        try:
            check(_lib.load().cb_timing_create(int(n), int(d), float(alpha), C.byref(self._h)))
        except CbError as e:
            if e.status == _lib.CB_ERR_INVALID_ARG and not 0.0 <= alpha <= 1.0:
                raise ValueError("InvalidRolloffError") from e
            raise

    def push(self, samples) -> float:
        x = np.ascontiguousarray(np.asarray(samples, dtype=np.complex128))
        est = C.c_double(0.0)
        check(_lib.load().cb_timing_push(self._h, _ptr(x), len(x), C.byref(est)))
        return est.value

    run = push

    def push_dev(self, d_samples: int, n: int, stream: int = 0) -> float:
        est = C.c_double(0.0)
        check(_lib.load().cb_timing_push_dev(self._h, d_samples, n, C.byref(est), stream))
        return est.value

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _lib.load().cb_timing_destroy(h)
            except Exception:
                pass


TimingEstimatorNode = TimingEstimator


def prn_bits(poly_mask: int, state: int, n: int, width: int = 8):
    """PrnGen::next_byte n times (src/prns.rs:64-71).  Returns (bits, new_state)."""
    st = C.c_uint64(state)
    out = np.empty(n, dtype=np.uint8)
    check(_lib.load().cb_prn_bits(poly_mask, C.byref(st), width, n, _ptr(out)))
    return out, st.value


def bits_to_symbols_dev(d_bits: int, nbits: int, mode: int, d_sym: int, stream: int = 0) -> int:
    m = _sz()
    check(_lib.load().cb_bits_to_symbols_dev(d_bits, nbits, mode, d_sym, C.byref(m), stream))
    return m.value


def quantize_i16_dev(d_in: int, nfloats: int, scale: float, d_out: int, stream: int = 0) -> None:
    check(_lib.load().cb_quantize_i16_dev(d_in, nfloats, scale, d_out, stream))


def synth_uniform_dev(seed: int, first: int, n: int, d_out: int, stream: int = 0) -> None:
    check(_lib.load().cb_synth_uniform_dev(seed, first, n, d_out, stream))
