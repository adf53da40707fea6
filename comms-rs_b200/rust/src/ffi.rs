//! Raw bindings of include/comms_b200.h (hand-written; the header is small and stable).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_float, c_int, c_uint, c_void};

macro_rules! opaque { ($($n:ident),*) => { $(#[repr(C)] pub struct $n { _p: [u8; 0] })* } }
opaque!(cb_stream, cb_buf, cb_fir, cb_mixer, cb_fft, cb_fm, cb_chain, cb_comm, cb_timing, cb_nco, cb_fir_f64, cb_fft_f64);

pub const CB_OK: c_int = 0;
pub const CB_ERR_INVALID_ARG: c_int = 1;
pub const CB_ERR_SIZE: c_int = 2;

extern "C" {
    pub fn cb_version() -> c_int;
    pub fn cb_last_error() -> *const c_char;
    pub fn cb_status_str(status: c_int) -> *const c_char;
    pub fn cb_device_count(count: *mut c_int) -> c_int;
    pub fn cb_init(device: c_int) -> c_int;
    pub fn cb_device_synchronize() -> c_int;
    pub fn cb_launch_count(count: *mut u64) -> c_int;

    pub fn cb_stream_create(out: *mut *mut cb_stream) -> c_int;
    pub fn cb_stream_destroy(s: *mut cb_stream) -> c_int;
    pub fn cb_stream_sync(s: *mut cb_stream) -> c_int;
    pub fn cb_stream_handle(s: *mut cb_stream) -> *mut c_void;

    pub fn cb_buf_alloc_pinned(bytes: usize, out: *mut *mut cb_buf) -> c_int;
    pub fn cb_buf_alloc_device(bytes: usize, out: *mut *mut cb_buf) -> c_int;
    pub fn cb_buf_retain(b: *mut cb_buf) -> c_int;
    pub fn cb_buf_release(b: *mut cb_buf) -> c_int;
    pub fn cb_buf_ptr(b: *mut cb_buf) -> *mut c_void;
    pub fn cb_buf_bytes(b: *mut cb_buf) -> usize;
    pub fn cb_buf_is_device(b: *mut cb_buf) -> c_int;
    pub fn cb_buf_record_ready(b: *mut cb_buf, stream: *mut c_void) -> c_int;
    pub fn cb_buf_wait_ready(b: *mut cb_buf, stream: *mut c_void) -> c_int;
    pub fn cb_buf_sync(b: *mut cb_buf) -> c_int;
    pub fn cb_copy_h2d_async(dst: *mut c_void, src: *const c_void, bytes: usize, stream: *mut c_void) -> c_int;
    pub fn cb_copy_d2h_async(dst: *mut c_void, src: *const c_void, bytes: usize, stream: *mut c_void) -> c_int;

    pub fn cb_fir_create(taps: *const c_float, ntaps: usize, state: *const c_float, nstate: usize,
                         decim: u32, interp: u32, out: *mut *mut cb_fir) -> c_int;
    pub fn cb_fir_destroy(h: *mut cb_fir) -> c_int;
    pub fn cb_fir_out_len(h: *const cb_fir, n_in: usize, n_out: *mut usize) -> c_int;
    pub fn cb_fir_run(h: *mut cb_fir, input: *const c_float, n_in: usize, out: *mut c_float, out_cap: usize,
                      n_out: *mut usize) -> c_int;
    pub fn cb_fir_run_dev(h: *mut cb_fir, d_in: *const c_float, n_in: usize, d_out: *mut c_float, out_cap: usize,
                          n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_fir_state_len(h: *const cb_fir, nstate: *mut usize) -> c_int;
    pub fn cb_fir_get_state(h: *mut cb_fir, state: *mut c_float, nstate: usize) -> c_int;
    pub fn cb_fir_set_state(h: *mut cb_fir, state: *const c_float, nstate: usize) -> c_int;
    pub fn cb_fir_stream(h: *mut cb_fir) -> *mut c_void;

    pub fn cb_fir_f64_create(taps: *const f64, ntaps: usize, state: *const f64, nstate: usize,
                             decim: u32, interp: u32, out: *mut *mut cb_fir_f64) -> c_int;
    pub fn cb_fir_f64_destroy(h: *mut cb_fir_f64) -> c_int;
    pub fn cb_fir_f64_out_len(h: *const cb_fir_f64, n_in: usize, n_out: *mut usize) -> c_int;
    pub fn cb_fir_f64_run(h: *mut cb_fir_f64, input: *const f64, n_in: usize, out: *mut f64, out_cap: usize,
                          n_out: *mut usize) -> c_int;
    pub fn cb_fir_f64_run_dev(h: *mut cb_fir_f64, d_in: *const f64, n_in: usize, d_out: *mut f64, out_cap: usize,
                              n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_fir_f64_state_len(h: *const cb_fir_f64, nstate: *mut usize) -> c_int;
    pub fn cb_fir_f64_get_state(h: *mut cb_fir_f64, state: *mut f64, nstate: usize) -> c_int;
    pub fn cb_fir_f64_set_state(h: *mut cb_fir_f64, state: *const f64, nstate: usize) -> c_int;
    pub fn cb_fir_f64_stream(h: *mut cb_fir_f64) -> *mut c_void;

    pub fn cb_decimate(input: *const c_void, n: usize, elem_bytes: usize, rate: usize, out: *mut c_void,
                       out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn cb_upsample(input: *const c_void, n: usize, elem_bytes: usize, rate: usize, out: *mut c_void,
                       out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn cb_decimate_dev(d_in: *const c_void, n: usize, elem_bytes: usize, rate: usize, d_out: *mut c_void,
                           out_cap: usize, n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_upsample_dev(d_in: *const c_void, n: usize, elem_bytes: usize, rate: usize, d_out: *mut c_void,
                           out_cap: usize, n_out: *mut usize, stream: *mut c_void) -> c_int;

    pub fn cb_mixer_create(dphase: c_double, phase: c_double, out: *mut *mut cb_mixer) -> c_int;
    pub fn cb_mixer_destroy(h: *mut cb_mixer) -> c_int;
    pub fn cb_mixer_run(h: *mut cb_mixer, input: *const c_float, n: usize, out: *mut c_float) -> c_int;
    pub fn cb_mixer_run_dev(h: *mut cb_mixer, d_in: *const c_float, n: usize, d_out: *mut c_float,
                            stream: *mut c_void) -> c_int;
    pub fn cb_mixer_get_phase(h: *const cb_mixer, phase: *mut c_double, dphase: *mut c_double) -> c_int;
    pub fn cb_mixer_set_phase(h: *mut cb_mixer, phase: c_double) -> c_int;

    pub fn cb_fft_create(fft_size: usize, inverse: c_int, out: *mut *mut cb_fft) -> c_int;
    pub fn cb_fft_destroy(h: *mut cb_fft) -> c_int;
    pub fn cb_fft_run(h: *mut cb_fft, input: *const c_float, n_in: usize, out: *mut c_float) -> c_int;
    pub fn cb_fft_run_dev(h: *mut cb_fft, d_in: *const c_float, n_in: usize, d_out: *mut c_float,
                          stream: *mut c_void) -> c_int;
    pub fn cb_fft_size(h: *const cb_fft, fft_size: *mut usize, inverse: *mut c_int) -> c_int;

    pub fn cb_fft_f64_create(fft_size: usize, inverse: c_int, out: *mut *mut cb_fft_f64) -> c_int;
    pub fn cb_fft_f64_destroy(h: *mut cb_fft_f64) -> c_int;
    pub fn cb_fft_f64_size(h: *const cb_fft_f64, fft_size: *mut usize, inverse: *mut c_int) -> c_int;
    pub fn cb_fft_f64_run(h: *mut cb_fft_f64, input: *const f64, n_in: usize, out: *mut f64) -> c_int;
    pub fn cb_fft_f64_run_dev(h: *mut cb_fft_f64, d_in: *const f64, n_in: usize, d_out: *mut f64,
                              stream: *mut c_void) -> c_int;

    pub fn cb_fm_create(out: *mut *mut cb_fm) -> c_int;
    pub fn cb_fm_destroy(h: *mut cb_fm) -> c_int;
    pub fn cb_fm_run(h: *mut cb_fm, input: *const c_float, n: usize, out: *mut c_float) -> c_int;
    pub fn cb_fm_run_dev(h: *mut cb_fm, d_in: *const c_float, n: usize, d_out: *mut c_float, stream: *mut c_void) -> c_int;

    pub fn cb_chain_create(channels: usize, dphase: *const c_double, phase: *const c_double, taps: *const c_float,
                           ntaps: usize, decim: u32, with_fm: c_int, out: *mut *mut cb_chain) -> c_int;
    pub fn cb_chain_destroy(h: *mut cb_chain) -> c_int;
    pub fn cb_chain_out_len(h: *const cb_chain, n_in: usize, n_out: *mut usize) -> c_int;
    pub fn cb_chain_run(h: *mut cb_chain, input: *const c_float, n_in: usize, out: *mut c_float, out_cap: usize,
                        n_out: *mut usize) -> c_int;
    pub fn cb_chain_run_dev(h: *mut cb_chain, d_in: *const c_float, n_in: usize, d_out: *mut c_float, out_cap: usize,
                            n_out: *mut usize, stream: *mut c_void) -> c_int;

    pub fn cb_fir_run_i16(h: *mut cb_fir, input: *const f32, n_in: usize, scale: f32, out: *mut i16, out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn cb_fir_run_dev_i16(h: *mut cb_fir, d_in: *const f32, n_in: usize, scale: f32, d_out: *mut i16, out_cap: usize, n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_convert_u8_dev(d_in: *const u8, n_samples: usize, d_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn cb_convert_i16_dev(d_in: *const i16, n_samples: usize, scale: f32, d_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn cb_chain_run_u8(h: *mut cb_chain, input: *const u8, n_in: usize, out: *mut f32, out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn cb_chain_run_u8_dev(h: *mut cb_chain, d_in: *const u8, n_in: usize, d_out: *mut f32, out_cap: usize, n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_comm_unique_id(id128: *mut c_void) -> c_int;
    pub fn cb_comm_init(nranks: c_int, rank: c_int, id128: *const c_void, out: *mut *mut cb_comm) -> c_int;
    pub fn cb_comm_destroy(c: *mut cb_comm) -> c_int;
    pub fn cb_gather_segments_dev(c: *mut cb_comm, d_seg: *const f32, n_samples: usize, d_all: *mut f32, stream: *mut c_void) -> c_int;
    pub fn cb_comm_rank(c: *const cb_comm, rank: *mut c_int, nranks: *mut c_int) -> c_int;
    pub fn cb_gather_segments_to_root_dev(c: *mut cb_comm, d_seg: *const c_void, counts: *const usize, elem_bytes: usize, root: c_int, d_all: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn cb_allgather_segments_var_dev(c: *mut cb_comm, d_seg: *const c_void, counts: *const usize, elem_bytes: usize, d_all: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn cb_peer_export(d_ptr: *mut c_void, handle64: *mut c_void) -> c_int;
    pub fn cb_peer_open(handle64: *const c_void, d_mapped: *mut *mut c_void) -> c_int;
    pub fn cb_peer_close(d_mapped: *mut c_void) -> c_int;
    pub fn cb_fir_run_iq16(h: *mut cb_fir, input: *const i16, n_in: usize, in_scale: f32, out_scale: f32, out: *mut i16, out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn cb_fir_run_dev_iq16(h: *mut cb_fir, d_in: *const i16, n_in: usize, in_scale: f32, out_scale: f32, d_out: *mut i16, out_cap: usize, n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_fft_run_iq16(h: *mut cb_fft, input: *const i16, n_in: usize, in_scale: f32, out: *mut f32) -> c_int;
    pub fn cb_fft_run_dev_iq16(h: *mut cb_fft, d_in: *const i16, n_in: usize, in_scale: f32, d_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn cb_pool_configure(is_device: c_int, max_live_bytes: usize, max_cached_bytes: usize, timeout_ms: c_int) -> c_int;
    pub fn cb_pool_stats(is_device: c_int, live_bytes: *mut usize, cached_bytes: *mut usize, hits: *mut u64, misses: *mut u64, waits: *mut u64) -> c_int;
    pub fn cb_pool_trim() -> c_int;
    pub fn cb_pool_throttle(timeout_ms: c_int) -> c_int;
    pub fn cb_buf_record_done(b: *mut cb_buf, stream: *mut c_void) -> c_int;
    pub fn cb_nco_create(dphase: f64, phase: f64, out: *mut *mut cb_nco) -> c_int;
    pub fn cb_nco_destroy(h: *mut cb_nco) -> c_int;
    pub fn cb_nco_run(h: *mut cb_nco, perr: *const f64, n: usize, out: *mut f64) -> c_int;
    pub fn cb_nco_run_dev(h: *mut cb_nco, d_perr: *const f64, n: usize, d_out: *mut f64, stream: *mut c_void) -> c_int;
    pub fn cb_nco_get_phase(h: *mut cb_nco, phase: *mut f64, dphase: *mut f64) -> c_int;
    pub fn cb_nco_set_phase(h: *mut cb_nco, phase: f64) -> c_int;
    pub fn cb_fir_run_real(h: *mut cb_fir, input: *const f32, n_in: usize, out: *mut f32, out_cap: usize, n_out: *mut usize) -> c_int;
    pub fn cb_fir_run_real_dev(h: *mut cb_fir, d_in: *const f32, n_in: usize, d_out: *mut f32, out_cap: usize, n_out: *mut usize, stream: *mut c_void) -> c_int;
    pub fn cb_qfilt_taps_f64(n_taps: u32, alpha: f64, sam_per_sym: u32, taps: *mut f64, n_out: *mut u32) -> c_int;
    pub fn cb_freq_estimate(samples: *const f64, n: usize, estimate: *mut f64) -> c_int;
    pub fn cb_freq_estimate_dev(d_samples: *const f64, n: usize, estimate: *mut f64, stream: *mut c_void) -> c_int;
    pub fn cb_timing_create(n: u32, d: u32, alpha: f64, out: *mut *mut cb_timing) -> c_int;
    pub fn cb_timing_destroy(h: *mut cb_timing) -> c_int;
    pub fn cb_timing_push(h: *mut cb_timing, samples: *const f64, n: usize, estimate: *mut f64) -> c_int;
    pub fn cb_timing_push_dev(h: *mut cb_timing, d_samples: *const f64, n: usize, estimate: *mut f64, stream: *mut c_void) -> c_int;
    pub fn cb_real_to_complex_dev(d_in: *const f32, n: usize, d_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn cb_complex_real_dev(d_in: *const f32, n: usize, d_out: *mut f32, stream: *mut c_void) -> c_int;
    pub fn cb_rrc_taps(n_taps: u32, sam_per_sym: f64, beta: f64, taps: *mut f32) -> c_int;
    pub fn cb_rrc_taps_f64(n_taps: u32, sam_per_sym: f64, beta: f64, taps: *mut f64) -> c_int;
    pub fn cb_prn_bits(poly_mask: u64, state: *mut u64, width: c_uint, n: usize, bits: *mut u8) -> c_int;
    pub fn cb_bits_to_symbols_dev(d_bits: *const u8, nbits: usize, mode: c_int, d_sym: *mut c_float, nsym: *mut usize,
                                  stream: *mut c_void) -> c_int;
    pub fn cb_quantize_i16_dev(d_in: *const c_float, nfloats: usize, scale: c_float, d_out: *mut i16,
                               stream: *mut c_void) -> c_int;
    pub fn cb_synth_uniform_dev(seed: u64, first: u64, n: usize, d_out: *mut c_float, stream: *mut c_void) -> c_int;
}
