"""comms-rs_b200: B200-native (sm_100a) implementation of comms-rs's FIR / mixer /
FFT hot path.  The product is libcomms_b200.so (csrc/, C ABI in
include/comms_b200.h); this package is the thin host-side mirror of the
reference's node structs used by tests and bench.  No CPU fallback exists.
"""
from . import _lib
from ._lib import CbError, NodeError, load
from .nodes import (BatchFirNode, BatchFirNodeF64, FirNodeF64, PulseNodeF64, ChainBank, DecimateNode, FFTBatchNode, FFTBatchNodeF64, FFTSampleNode, FFTSampleNodeF64, FirNode, FMDemodNode,
                    MixerNode, NcoNode, PulseNode, UpsampleNode, bits_to_symbols_dev, complex_real_dev, convert_i16_dev, convert_u8_dev,
                    prn_bits, real_to_complex_dev,
                    quantize_i16_dev,
                    rrc_taps, synth_uniform_dev, TimingEstimator, TimingEstimatorNode, frequency_offset_estimate,
                    frequency_offset_estimate_dev, qfilt_taps)


def init(device: int = 0) -> None:
    """cb_init: bind this thread to `device`; raises CbError(NO_DEVICE) without a GPU."""
    _lib.check(load().cb_init(device))


def device_count() -> int:
    import ctypes as C
    n = C.c_int()
    _lib.check(load().cb_device_count(C.byref(n)))
    return n.value


def synchronize() -> None:
    _lib.check(load().cb_device_synchronize())


def launch_count() -> int:
    """Kernels launched by libcomms_b200 in this process so far (cb_launch_count)."""
    import ctypes as C
    n = C.c_uint64()
    _lib.check(load().cb_launch_count(C.byref(n)))
    return n.value



def pool_configure(is_device: bool, max_live_bytes: int = 0, max_cached_bytes: int = 1 << 30, timeout_ms: int = 10000) -> None:
    """cb_pool_configure: high-water mark (back-pressure), cache size and blocking timeout of the buffer pool."""
    _lib.check(load().cb_pool_configure(int(bool(is_device)), int(max_live_bytes), int(max_cached_bytes), int(timeout_ms)))


def pool_stats(is_device: bool) -> dict:
    import ctypes as C
    live, cached = C.c_size_t(), C.c_size_t()
    hits, misses, waits = C.c_uint64(), C.c_uint64(), C.c_uint64()
    _lib.check(load().cb_pool_stats(int(bool(is_device)), C.byref(live), C.byref(cached), C.byref(hits), C.byref(misses), C.byref(waits)))
    return {"live_bytes": live.value, "cached_bytes": cached.value, "hits": hits.value, "misses": misses.value, "waits": waits.value}


from . import sharding  # noqa: E402
