"""ctypes binding of libcomms_b200.so (include/comms_b200.h).

The library is the product; this module only declares its entry points.  There
is no fallback of any kind: if the shared library is missing, or a compute call
is made without a CUDA device, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcomms_b200.so")

CB_OK, CB_ERR_INVALID_ARG, CB_ERR_SIZE, CB_ERR_CUDA, CB_ERR_NO_DEVICE, CB_ERR_OOM, CB_ERR_UNSUPPORTED = range(7)


class CbError(RuntimeError):
    """A non-zero cb_status.  `.status` holds the code; the Rust shim would map
    INVALID_ARG / SIZE to NodeError::DataError and the rest to PermanentError."""

    def __init__(self, status: int, message: str):
        super().__init__(f"libcomms_b200 status {status}: {message}")
        self.status = status


class NodeError(Exception):
    """Mirror of NodeError (src/node/mod.rs:68-73)."""

    DataError = "DataError"
    PermanentError = "PermanentError"
    DataEnd = "DataEnd"
    CommError = "CommError"

    def __init__(self, kind: str, detail: str = ""):
        super().__init__(f"{kind}: {detail}" if detail else kind)
        self.kind = kind


_vp, _sz, _u32, _i, _dbl = C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, C.c_double
_pp = C.POINTER(C.c_void_p)
_psz = C.POINTER(C.c_size_t)

# name -> (restype, argtypes); every symbol include/comms_b200.h declares
SIGNATURES = {
    "cb_version": (_i, []),
    "cb_last_error": (C.c_char_p, []),
    "cb_status_str": (C.c_char_p, [_i]),
    "cb_device_count": (_i, [C.POINTER(_i)]),
    "cb_init": (_i, [_i]),
    "cb_device_synchronize": (_i, []),
    "cb_launch_count": (_i, [C.POINTER(C.c_uint64)]),
    "cb_stream_create": (_i, [_pp]),
    "cb_stream_destroy": (_i, [_vp]),
    "cb_stream_sync": (_i, [_vp]),
    "cb_stream_handle": (_vp, [_vp]),
    "cb_buf_alloc_pinned": (_i, [_sz, _pp]),
    "cb_buf_alloc_device": (_i, [_sz, _pp]),
    "cb_pool_configure": (_i, [_i, _sz, _sz, _i]),
    "cb_pool_stats": (_i, [_i, _psz, _psz, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "cb_pool_trim": (_i, []),
    "cb_pool_throttle": (_i, [_i]),
    "cb_buf_record_done": (_i, [_vp, _vp]),
    "cb_buf_retain": (_i, [_vp]),
    "cb_buf_release": (_i, [_vp]),
    "cb_buf_ptr": (_vp, [_vp]),
    "cb_buf_bytes": (_sz, [_vp]),
    "cb_buf_is_device": (_i, [_vp]),
    "cb_buf_record_ready": (_i, [_vp, _vp]),
    "cb_buf_wait_ready": (_i, [_vp, _vp]),
    "cb_buf_sync": (_i, [_vp]),
    "cb_copy_h2d_async": (_i, [_vp, _vp, _sz, _vp]),
    "cb_copy_d2h_async": (_i, [_vp, _vp, _sz, _vp]),
    "cb_fir_create": (_i, [_vp, _sz, _vp, _sz, _u32, _u32, _pp]),
    "cb_fir_destroy": (_i, [_vp]),
    "cb_fir_out_len": (_i, [_vp, _sz, _psz]),
    "cb_fir_run": (_i, [_vp, _vp, _sz, _vp, _sz, _psz]),
    "cb_fir_run_dev": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp]),
    "cb_fir_run_real": (_i, [_vp, _vp, _sz, _vp, _sz, _psz]),
    "cb_fir_run_real_dev": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp]),
    "cb_fir_run_i16": (_i, [_vp, _vp, _sz, C.c_float, _vp, _sz, C.POINTER(_sz)]),
    "cb_fir_run_dev_i16": (_i, [_vp, _vp, _sz, C.c_float, _vp, _sz, C.POINTER(_sz), _vp]),
    "cb_fir_run_iq16": (_i, [_vp, _vp, _sz, C.c_float, C.c_float, _vp, _sz, _psz]),
    "cb_fir_run_dev_iq16": (_i, [_vp, _vp, _sz, C.c_float, C.c_float, _vp, _sz, _psz, _vp]),
    "cb_fft_run_iq16": (_i, [_vp, _vp, _sz, C.c_float, _vp]),
    "cb_fft_run_dev_iq16": (_i, [_vp, _vp, _sz, C.c_float, _vp, _vp]),
    "cb_fir_state_len": (_i, [_vp, _psz]),
    "cb_fir_get_state": (_i, [_vp, _vp, _sz]),
    "cb_fir_set_state": (_i, [_vp, _vp, _sz]),
    "cb_fir_stream": (_vp, [_vp]),
    "cb_fir_f64_create": (_i, [_vp, _sz, _vp, _sz, _u32, _u32, _pp]),
    "cb_fir_f64_destroy": (_i, [_vp]),
    "cb_fir_f64_out_len": (_i, [_vp, _sz, _psz]),
    "cb_fir_f64_run": (_i, [_vp, _vp, _sz, _vp, _sz, _psz]),
    "cb_fir_f64_run_dev": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp]),
    "cb_fir_f64_state_len": (_i, [_vp, _psz]),
    "cb_fir_f64_get_state": (_i, [_vp, _vp, _sz]),
    "cb_fir_f64_set_state": (_i, [_vp, _vp, _sz]),
    "cb_fir_f64_stream": (_vp, [_vp]),
    "cb_fft_f64_create": (_i, [_sz, _i, _pp]),
    "cb_fft_f64_destroy": (_i, [_vp]),
    "cb_fft_f64_size": (_i, [_vp, _psz, C.POINTER(_i)]),
    "cb_fft_f64_run": (_i, [_vp, _vp, _sz, _vp]),
    "cb_fft_f64_run_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "cb_decimate_dev": (_i, [_vp, _sz, _sz, _sz, _vp, _sz, _psz, _vp]),
    "cb_upsample_dev": (_i, [_vp, _sz, _sz, _sz, _vp, _sz, _psz, _vp]),
    "cb_decimate": (_i, [_vp, _sz, _sz, _sz, _vp, _sz, _psz]),
    "cb_upsample": (_i, [_vp, _sz, _sz, _sz, _vp, _sz, _psz]),
    "cb_mixer_create": (_i, [_dbl, _dbl, _pp]),
    "cb_mixer_destroy": (_i, [_vp]),
    "cb_mixer_run": (_i, [_vp, _vp, _sz, _vp]),
    "cb_mixer_run_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "cb_mixer_get_phase": (_i, [_vp, C.POINTER(_dbl), C.POINTER(_dbl)]),
    "cb_mixer_set_phase": (_i, [_vp, _dbl]),
    "cb_fft_create": (_i, [_sz, _i, _pp]),
    "cb_fft_destroy": (_i, [_vp]),
    "cb_fft_run": (_i, [_vp, _vp, _sz, _vp]),
    "cb_fft_run_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "cb_fft_size": (_i, [_vp, _psz, C.POINTER(_i)]),
    "cb_fm_create": (_i, [_pp]),
    "cb_fm_destroy": (_i, [_vp]),
    "cb_fm_run": (_i, [_vp, _vp, _sz, _vp]),
    "cb_fm_run_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "cb_chain_create": (_i, [_sz, _vp, _vp, _vp, _sz, _u32, _i, _pp]),
    "cb_chain_destroy": (_i, [_vp]),
    "cb_chain_out_len": (_i, [_vp, _sz, _psz]),
    "cb_chain_run": (_i, [_vp, _vp, _sz, _vp, _sz, _psz]),
    "cb_chain_run_dev": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp]),
    "cb_chain_run_u8_dev": (_i, [_vp, _vp, _sz, _vp, _sz, _psz, _vp]),
    "cb_chain_run_u8": (_i, [_vp, _vp, _sz, _vp, _sz, _psz]),
    "cb_comm_unique_id": (_i, [_vp]),
    "cb_comm_init": (_i, [C.c_int, C.c_int, _vp, C.POINTER(_vp)]),
    "cb_comm_destroy": (_i, [_vp]),
    "cb_gather_segments_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "cb_comm_rank": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
    "cb_gather_segments_to_root_dev": (_i, [_vp, _vp, _psz, _sz, _i, _vp, _vp]),
    "cb_allgather_segments_var_dev": (_i, [_vp, _vp, _psz, _sz, _vp, _vp]),
    "cb_peer_export": (_i, [_vp, _vp]),
    "cb_peer_open": (_i, [_vp, _pp]),
    "cb_peer_close": (_i, [_vp]),
    "cb_real_to_complex_dev": (_i, [_vp, _sz, _vp, _vp]),
    "cb_complex_real_dev": (_i, [_vp, _sz, _vp, _vp]),
    "cb_convert_u8_dev": (_i, [_vp, _sz, _vp, _vp]),
    "cb_convert_i16_dev": (_i, [_vp, _sz, C.c_float, _vp, _vp]),
    "cb_qfilt_taps_f64": (_i, [_u32, _dbl, _u32, _vp, C.POINTER(_u32)]),
    "cb_freq_estimate": (_i, [_vp, _sz, C.POINTER(_dbl)]),
    "cb_freq_estimate_dev": (_i, [_vp, _sz, C.POINTER(_dbl), _vp]),
    "cb_timing_create": (_i, [_u32, _u32, _dbl, _pp]),
    "cb_timing_destroy": (_i, [_vp]),
    "cb_timing_push": (_i, [_vp, _vp, _sz, C.POINTER(_dbl)]),
    "cb_timing_push_dev": (_i, [_vp, _vp, _sz, C.POINTER(_dbl), _vp]),
    "cb_nco_create": (_i, [_dbl, _dbl, _pp]),
    "cb_nco_destroy": (_i, [_vp]),
    "cb_nco_run": (_i, [_vp, _vp, _sz, _vp]),
    "cb_nco_run_dev": (_i, [_vp, _vp, _sz, _vp, _vp]),
    "cb_nco_get_phase": (_i, [_vp, C.POINTER(_dbl), C.POINTER(_dbl)]),
    "cb_nco_set_phase": (_i, [_vp, _dbl]),
    "cb_rrc_taps": (_i, [C.c_uint32, C.c_double, C.c_double, _vp]),
    "cb_rrc_taps_f64": (_i, [C.c_uint32, C.c_double, C.c_double, _vp]),
    "cb_prn_bits": (_i, [C.c_uint64, C.POINTER(C.c_uint64), C.c_uint, _sz, _vp]),
    "cb_bits_to_symbols_dev": (_i, [_vp, _sz, _i, _vp, _psz, _vp]),
    "cb_quantize_i16_dev": (_i, [_vp, _sz, C.c_float, _vp, _vp]),
    "cb_synth_uniform_dev": (_i, [C.c_uint64, C.c_uint64, _sz, _vp, _vp]),
}

_LIB = None


def load() -> C.CDLL:
    """dlopen libcomms_b200.so and type every entry point.  Raises if the
    library has not been built (python comms-rs_b200/build.py) -- loudly, on
    purpose: nothing else can stand in for it."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python comms-rs_b200/build.py` "
                "(nvcc, sm_100a).  There is no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the header and the .so disagree
            fn.restype, fn.argtypes = res, args
        _LIB = lib
    return _LIB


def check(status: int) -> None:
    if status != CB_OK:
        msg = load().cb_last_error().decode(errors="replace")
        raise CbError(status, msg or load().cb_status_str(status).decode())


def node_error(e: CbError) -> NodeError:
    kind = NodeError.DataError if e.status in (CB_ERR_INVALID_ARG, CB_ERR_SIZE) else NodeError.PermanentError
    return NodeError(kind, str(e))
