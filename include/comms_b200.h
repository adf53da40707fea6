/*
 * comms_b200.h -- C ABI of libcomms_b200.so, the B200 (sm_100a) implementation
 * of comms-rs's FIR / mixer / FFT hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.
 * A `Complex<f32>` slice (`#[repr(C)] {re, im}`) crosses as `const float*`
 * holding 2*n interleaved floats; lengths are in complex samples unless the
 * name says otherwise.  Each entry point cites the reference item (path:line in
 * ostrosco/comms-rs) it replaces; INTEGRATION.md shows the Rust binding.
 *
 * Conventions
 *   - every function returns a cb_status (0 = ok) and never throws or aborts;
 *     cb_last_error() gives the calling thread's last message.
 *     Suggested mapping in the Rust shim: CB_ERR_INVALID_ARG / CB_ERR_SIZE ->
 *     NodeError::DataError, everything else -> NodeError::PermanentError
 *     (src/node/mod.rs:68-73).
 *   - handles are used by one thread at a time (Node: Send, not Sync;
 *     src/node/mod.rs:94) but different handles may be used concurrently from
 *     different threads: the library keeps no unsynchronised global state,
 *     sets the device per call and gives each handle its own non-blocking
 *     stream.
 *   - `*_run` (host pointers) has Vec-in / Vec-out semantics: it returns when
 *     `out` is filled.  `*_run_dev` takes device pointers (16-byte aligned for
 *     full speed) and a cudaStream_t (NULL = the handle's stream), is
 *     asynchronous, and lets nodes chain on the device.
 *   - input and output ranges of a `*_run_dev` call must not overlap
 *     (CB_ERR_INVALID_ARG): the filter, chain, FM and FFT kernels read samples
 *     owned by neighbouring tiles and rebuild the carried state from the input.
 *     Only the element-wise entries (mixer, converters, quantiser) may run
 *     in place.
 *   - a handle's carried state is ordered across streams: each `*_run_dev`
 *     records an event behind its launch and the handle's next use on any other
 *     stream (and get/set_state, destroy) waits for it, so calls on different
 *     streams behave like calls on one stream, in host call order.
 *   - there is no CPU fallback: without a CUDA device every compute call
 *     fails with CB_ERR_NO_DEVICE.
 */
#ifndef COMMS_B200_H
#define COMMS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define CB_API
#else
#define CB_API __attribute__((visibility("default")))
#endif

typedef enum cb_status {
    CB_OK = 0,
    CB_ERR_INVALID_ARG = 1, /* null pointer, zero fft size, bad rate ...      */
    CB_ERR_SIZE = 2,        /* input length does not fit (e.g. len != fft_size,
                               out_cap too small)                             */
    CB_ERR_CUDA = 3,        /* a CUDA runtime call failed                     */
    CB_ERR_NO_DEVICE = 4,   /* no usable CUDA device / cb_init not possible   */
    CB_ERR_OOM = 5,         /* host or device allocation failed               */
    CB_ERR_UNSUPPORTED = 6  /* valid in the reference, not provided here      */
} cb_status;

typedef struct cb_stream cb_stream;   /* a device + cudaStream_t                  */
typedef struct cb_buf cb_buf;         /* ref-counted pinned-host or device buffer */
typedef struct cb_fir cb_fir;         /* BatchFirNode / FirNode / PulseNode state */
typedef struct cb_mixer cb_mixer;     /* Mixer state                              */
typedef struct cb_fft cb_fft;         /* BatchFFT plan                            */
typedef struct cb_fm cb_fm;           /* FM demod state                           */
typedef struct cb_chain cb_chain;     /* bank of fused mixer->FIR->decimate->FM   */

/* ------------------------------------------------------------------ library */
CB_API int cb_version(void);                       /* 1000*major + minor        */
CB_API const char *cb_last_error(void);            /* thread-local, never NULL  */
CB_API const char *cb_status_str(int status);
CB_API int cb_device_count(int *count);
/* Binds the calling thread's subsequent creates to `device` (default 0). */
CB_API int cb_init(int device);
CB_API int cb_device_synchronize(void);
/* Number of CUDA kernels this library has launched in the process so far (a
 * metrics hook with no reference counterpart; bench.py reports it as
 * gpu_launches). */
CB_API int cb_launch_count(uint64_t *count);

/* ------------------------------------------------------------------ streams */
CB_API int cb_stream_create(cb_stream **out);
CB_API int cb_stream_destroy(cb_stream *s);
CB_API int cb_stream_sync(cb_stream *s);
CB_API void *cb_stream_handle(cb_stream *s);       /* the cudaStream_t          */

/* ------------------------------------------------------------------ buffers
 * What crosses a NodeSender/NodeReceiver channel instead of a Vec when two GPU
 * nodes are adjacent: the derive macro clones the result once per downstream
 * edge (node_derive/src/lib.rs:156), so Clone must be cb_buf_retain, Drop
 * cb_buf_release. */
/* Blocks come from a size-classed, thread-safe pool per (device, kind): no cudaMalloc / cudaFree per message.  The
 * pool applies BACK-PRESSURE for the reference's unbounded channels (src/node/mod.rs:152; Graph::new(Some(n)),
 * src/node/graph.rs:44-47, is the bounded alternative): with a high-water mark set (cb_pool_configure), the nodes where
 * pool buffers START (a source filling pinned messages, a host->device edge node) call cb_pool_throttle() once per
 * message: it blocks while the bytes handed out and not yet released exceed the mark of either kind, and fails with
 * CB_ERR_OOM after timeout_ms (<= 0: the configured default) if no consumer releases.  Allocations themselves never
 * block -- a node that waited for a buffer while holding one could close a cycle of waits.
 * max_live_bytes = 0: no mark (default); max_cached_bytes: released blocks kept for reuse (default 1 GiB).
 * A consumer that launched asynchronous work on a buffer calls cb_buf_record_done(buf, its stream) before dropping its
 * reference; the pool waits for those events (and the producer's ready event) before the block's next owner gets it. */
CB_API int cb_pool_configure(int is_device, size_t max_live_bytes, size_t max_cached_bytes, int timeout_ms);
CB_API int cb_pool_stats(int is_device, size_t *live_bytes, size_t *cached_bytes, uint64_t *hits, uint64_t *misses,
                         uint64_t *waits);
CB_API int cb_pool_trim(void);
CB_API int cb_pool_throttle(int timeout_ms);
CB_API int cb_buf_record_done(cb_buf *b, void *stream);
CB_API int cb_buf_alloc_pinned(size_t bytes, cb_buf **out);
CB_API int cb_buf_alloc_device(size_t bytes, cb_buf **out);
CB_API int cb_buf_retain(cb_buf *b);
CB_API int cb_buf_release(cb_buf *b);
CB_API void *cb_buf_ptr(cb_buf *b);
CB_API size_t cb_buf_bytes(cb_buf *b);
CB_API int cb_buf_is_device(cb_buf *b);
/* Hand-off between nodes on different streams without a host sync: the producer
 * records "content complete" on its stream, the consumer makes its stream wait
 * (no-op if nothing was recorded); cb_buf_sync blocks the host until ready. */
CB_API int cb_buf_record_ready(cb_buf *b, void *stream);
CB_API int cb_buf_wait_ready(cb_buf *b, void *stream);
CB_API int cb_buf_sync(cb_buf *b);
/* async copies on `stream` (NULL = default stream of the bound device) */
CB_API int cb_copy_h2d_async(void *dst_dev, const void *src_host, size_t bytes, void *stream);
CB_API int cb_copy_d2h_async(void *dst_host, const void *src_dev, size_t bytes, void *stream);

/* ------------------------------------------------------------------ FIR
 * Replaces batch_fir / fir (src/filter/fir.rs:87-102, :43-54) and the state
 * handling of BatchFirNode::new / FirNode::new (src/filter/fir_node.rs:193-211):
 *   y[n] = sum_{k < min(ntaps, nstate)} taps[k] * x[n-k],  x[-1-k] = state[k].
 * `state` may be NULL (zeros of length ntaps, like `None`); otherwise nstate
 * complex samples, newest first.  The state is carried across calls, so batch
 * boundaries are invisible in the output stream.
 *
 * decim / interp fuse the neighbouring resample nodes:
 *   interp = L > 1: input is zero-stuffed by L first (UpsampleNode::upsample,
 *     src/util/resample_node.rs:120-131, or PulseNode::run, src/pulse.rs:82-92)
 *     -- computed as a polyphase bank, n inputs -> n*L outputs;
 *   decim = D > 1: only outputs 0, D, 2D.. OF EACH CALL survive
 *     (DecimateNode::decimate, src/util/resample_node.rs:53-65; the phase is
 *     reset per batch, as in the reference) -> ceil(n*L / D) outputs.
 *   0 and 1 both mean pass-through, as in the reference.
 * With interp > 1 an explicit initial `state` must be consistent with a
 * zero-stuffed history (non-zero only every L-th entry, newest = index L-1
 * ... ) or be NULL; otherwise CB_ERR_UNSUPPORTED.
 */
/* Numerical locality.  Filters of up to 128 taps (and the polyphase banks) keep the reference's locality per output:
 * every output y[n] is within 1e-5 * sum_k |taps[k]| |x[n-k]| of the exact value -- a quiet stretch next to a loud
 * one keeps its own accuracy -- and an Inf / NaN input sample makes exactly the outputs non-finite whose taps reach it
 * (tiles the tensor-core kernels cannot hold to that are recomputed in plain f32).  One exception: the tensor-core
 * kernels split the taps with one scale, so a tap far below the largest is carried to ~2^-39 of the largest tap in
 * absolute terms (an impulse through a tap of 1e-8 of the largest is off by ~1e-4 of itself); with any dense input
 * this is far below f32 rounding.  The
 * fast-convolution path for 129..1025 taps (calls of >= 8192 samples) works on frames of 4096 points: its error is
 * relative to the frame's energy: every output of frame f is within (2 rho_4096 + 2^-24) * max_k |H_k| * ||x_f||_2
 * of the exact value (rho_4096 = 1.6 * 12 * 2^-24, the FFT's norm bound below; H the 4096-point transform of the taps;
 * x_f the frame's 4096 inputs, history included), and one non-finite sample makes the outputs of exactly the frames
 * whose 4096 inputs hold it non-finite.  COMMS_B200_FIR_PATH=cuda selects the direct form for such filters when that matters. */
CB_API int cb_fir_create(const float *taps, size_t ntaps, const float *state, size_t nstate,
                         uint32_t decim, uint32_t interp, cb_fir **out);
CB_API int cb_fir_destroy(cb_fir *h);
CB_API int cb_fir_out_len(const cb_fir *h, size_t n_in, size_t *n_out);
CB_API int cb_fir_run(cb_fir *h, const float *in, size_t n_in, float *out, size_t out_cap, size_t *n_out);
CB_API int cb_fir_run_dev(cb_fir *h, const float *d_in, size_t n_in, float *d_out, size_t out_cap,
                          size_t *n_out, void *stream);
/* state as the reference would hold it after the samples seen so far
 * (newest first, nstate entries, in the zero-stuffed domain when interp > 1) */
/* Same filter step with the example's output quantiser fused behind it
 * (examples/single_thread_bpsk.rs:40-48: `(8192.0 * x) as i16`, written as the
 * interleaved native-endian i16 IQ stream of src/io/raw_iq.rs:185-223):
 * d_out receives 2*n_out int16 (re, im).  Polyphase interpolators on the
 * tensor-core path quantise in their epilogue (4 instead of 8 bytes written
 * per sample); every other shape filters into an internal f32 scratch and
 * runs the stand-alone quantiser.  Results are identical either way. */
CB_API int cb_fir_run_dev_i16(cb_fir *h, const float *d_in, size_t n_in, float scale, int16_t *d_out,
                              size_t out_cap, size_t *n_out, void *stream);
CB_API int cb_fir_run_i16(cb_fir *h, const float *in, size_t n_in, float scale, int16_t *out, size_t out_cap,
                          size_t *n_out);
/* i16 IQ on both edges -- what IQBatchInput / IQBatchOutput read and write (src/io/raw_iq.rs:78-140, 185-223:
 * interleaved native-endian i16): x = in_scale * (i16 as f32) (in_scale = 1: the plain cast of a
 * Vec<Complex<i16>>), this filter, out = (out_scale * y) as i16 (truncating, saturating).  d_in / in: 2*n_in int16,
 * d_out / out: 2*n_out int16.  Results are identical to cb_convert_i16 -> cb_fir_run -> cb_quantize_i16; every edge
 * carries 4 instead of 8 bytes per sample (the host-pointer form is PCIe-bound: twice the samples per second).
 * Plain filters of up to 128 taps on long batches run as ONE kernel that reads and writes the i16 words itself
 * (tensor-core FIR, fir_tc_kernel.cu IQ16; 16-byte aligned d_in); other shapes widen, filter and quantise in turn. */
CB_API int cb_fir_run_dev_iq16(cb_fir *h, const int16_t *d_in, size_t n_in, float in_scale, float out_scale,
                               int16_t *d_out, size_t out_cap, size_t *n_out, void *stream);
CB_API int cb_fir_run_iq16(cb_fir *h, const int16_t *in, size_t n_in, float in_scale, float out_scale, int16_t *out,
                           size_t out_cap, size_t *n_out);
/* Real samples in, real parts out: x -> Complex(x, 0) -> this filter -> .re, i.e. Convert2Node -> BatchFirNode ->
 * Convert3Node [-> DecimateNode] of examples/fm_radio.rs:98-164 in one call (n_in floats in, *n_out floats out; same
 * state, sizes and errors as cb_fir_run).  Fused into one kernel for <= 64 taps and decim in {2, 4, 5, 8, 10}. */
CB_API int cb_fir_run_real(cb_fir *h, const float *in, size_t n_in, float *out, size_t out_cap, size_t *n_out);
CB_API int cb_fir_run_real_dev(cb_fir *h, const float *d_in, size_t n_in, float *d_out, size_t out_cap, size_t *n_out,
                               void *stream);
CB_API int cb_fir_state_len(const cb_fir *h, size_t *nstate);
CB_API int cb_fir_get_state(cb_fir *h, float *state, size_t nstate);
CB_API int cb_fir_set_state(cb_fir *h, const float *state, size_t nstate);
CB_API void *cb_fir_stream(cb_fir *h);

/* ------------------------------------------------------------------ resample
 * Stand-alone DecimateNode::decimate / UpsampleNode::upsample
 * (src/util/resample_node.rs:53-65, :120-131) for graphs that keep them as
 * separate nodes.  elem_bytes = size of T (4, 8 or 16).  Device pointers. */
CB_API int cb_decimate_dev(const void *d_in, size_t n, size_t elem_bytes, size_t rate, void *d_out,
                           size_t out_cap, size_t *n_out, void *stream);
CB_API int cb_upsample_dev(const void *d_in, size_t n, size_t elem_bytes, size_t rate, void *d_out,
                           size_t out_cap, size_t *n_out, void *stream);
CB_API int cb_decimate(const void *in, size_t n, size_t elem_bytes, size_t rate, void *out,
                       size_t out_cap, size_t *n_out);
CB_API int cb_upsample(const void *in, size_t n, size_t elem_bytes, size_t rate, void *out,
                       size_t out_cap, size_t *n_out);

/* ------------------------------------------------------------------ mixer
 * Replaces Mixer::new / Mixer::mix (src/mixer.rs:43-51, :73-84) over a batch:
 *   y[n] = x[n] * exp(j*(phase + n*dphase)),  dphase wrapped into [0, 2pi)
 * Phase arithmetic in f64, carried across calls.  Note the argument order of
 * MixerNode::new(dphase, phase) (src/mixer.rs:128).
 * Accuracy, every output n counted from the stream's start (u32 = 2^-24, u64 = 2^-53, theta_n the exact phase):
 *   |y[n] - x[n] exp(j theta_n)| <= (13 u32 + u64 (|phase| + n dphase + 8 pi + c)) |x[n]| + 2^-148,
 * with c = sum over earlier calls of (2 pi + 2^-9 (|phase entering the call| + its length * dphase)) for the carried
 * phase.  13 u32 comes from sincosf's 2 ulp, the hi/lo correction and two fused complex products.  x[n] = 0 gives an
 * exact 0; a non-finite x[n] gives a non-finite y[n] and leaves every other output unchanged.
 * (tests/test_gpu_phase_bounds.py checks every output.) */
CB_API int cb_mixer_create(double dphase, double phase, cb_mixer **out);
CB_API int cb_mixer_destroy(cb_mixer *h);
CB_API int cb_mixer_run(cb_mixer *h, const float *in, size_t n, float *out);
CB_API int cb_mixer_run_dev(cb_mixer *h, const float *d_in, size_t n, float *d_out, void *stream);
CB_API int cb_mixer_get_phase(const cb_mixer *h, double *phase, double *dphase);
CB_API int cb_mixer_set_phase(cb_mixer *h, double phase);

/* ------------------------------------------------------------------ FFT
 * Replaces BatchFFT::run_fft (src/fft/mod.rs:73-96) / FFTBatchNode::new
 * (src/fft/fft_node.rs:65-74): X[k] = sum_n x[n] exp(-/+ j 2 pi k n / N),
 * "+" when inverse != 0, no 1/N in either direction, any N >= 1: powers of
 * two up to 2^20, any other length up to 2^19 (chirp-z above 128 points);
 * beyond that cb_fft_create returns CB_ERR_UNSUPPORTED.
 * n_in must be a multiple of fft_size (the reference requires n_in ==
 * fft_size, one frame per message; several contiguous frames per call is the
 * batched form) else CB_ERR_SIZE.
 * Numerical contract, per frame f of N points with S_f = sum_n |x[n]|, u = 2^-24 and X the exact transform: every
 * bin satisfies |X'[k] - X[k]| <= tau * S_f (+ 4 N 2^-149 for subnormal frames) and the frame
 * ||X' - X||_2 <= rho * ||X||_2, with
 *   powers of two (8 .. 2^20):       tau = 4 log2(N) u,    rho = 1.6 log2(N) u  (<= 2e-6 at every size)
 *   direct O(N^2) sums (N <= 128):   tau = rho = 5 u, whatever N
 *   chirp-z (M = padded power of two, the least >= max(256, 2N - 1)):
 *                                    tau = 5.4 log2(M) u,  rho = 2 log2(M) u.
 * A frame of zeros gives exact zeros.  A non-finite input makes every bin of its own frame non-finite and no other:
 * the other frames of the batch keep their bounds (tests/test_gpu_fft_bounds.py checks every bin of every plan). */
CB_API int cb_fft_create(size_t fft_size, int inverse, cb_fft **out);
CB_API int cb_fft_destroy(cb_fft *h);
CB_API int cb_fft_run(cb_fft *h, const float *in, size_t n_in, float *out);
CB_API int cb_fft_run_dev(cb_fft *h, const float *d_in, size_t n_in, float *d_out, void *stream);
CB_API int cb_fft_size(const cb_fft *h, size_t *fft_size, int *inverse);
/* i16 IQ frames in (IQBatchInput, src/io/raw_iq.rs:78-140): x = in_scale * (i16 as f32); complex f32 spectra out.
 * Power-of-two sizes up to 2^14 and 65536 points widen the samples in the transform's first loads (no extra pass);
 * spectra are bit-identical to cb_convert_i16 -> cb_fft_run. */
CB_API int cb_fft_run_iq16(cb_fft *h, const int16_t *in, size_t n_in, float in_scale, float *out);
CB_API int cb_fft_run_dev_iq16(cb_fft *h, const int16_t *d_in, size_t n_in, float in_scale, float *d_out, void *stream);

/* ------------------------------------------------------------------ FM demod
 * Replaces FM::demod (src/modulation/analog.rs:22-34): out[n] =
 * arg(x[n] * conj(x[n-1])), previous sample carried across calls, initially 0
 * (src/modulation/analog.rs:43-47).  n complex in -> n floats out. */
CB_API int cb_fm_create(cb_fm **out);
CB_API int cb_fm_destroy(cb_fm *h);
CB_API int cb_fm_run(cb_fm *h, const float *in, size_t n, float *out);
CB_API int cb_fm_run_dev(cb_fm *h, const float *d_in, size_t n, float *d_out, void *stream);

/* ------------------------------------------------------------------ fused bank
 * `channels` independent instances of
 *   [MixerNode] -> BatchFirNode -> DecimateNode(D) -> [FMDemodNode]
 * (the fm_radio front end, examples/fm_radio.rs:144-164, generalised per
 * BASELINE config 4) in ONE kernel that writes only the surviving samples.
 * Per channel c the semantics are exactly the four reference nodes in series,
 * each with its own carried state (mixer phase, FIR delay line, FM prev); the
 * decimation phase restarts at every call, like DecimateNode.
 * Layout: in  = channels x n_in complex, channel-major (channel c at
 *               in + 2*c*n_in floats);
 *         out = channels x ceil(n_in/D) floats (with_fm) or complex (no fm).
 * dphase/phase: per-channel arrays (NULL => mixer stage absent).
 * Taps are shared by all channels. */
CB_API int cb_chain_create(size_t channels, const double *dphase, const double *phase,
                           const float *taps, size_t ntaps, uint32_t decim, int with_fm,
                           cb_chain **out);
CB_API int cb_chain_destroy(cb_chain *h);
CB_API int cb_chain_out_len(const cb_chain *h, size_t n_in, size_t *n_out_per_channel);
CB_API int cb_chain_run(cb_chain *h, const float *in, size_t n_in, float *out, size_t out_cap_per_channel,
                        size_t *n_out_per_channel);
/* Same bank fed with the raw RTL-SDR byte stream (channel-major, n_in byte pairs per channel): ConvertNode
 * (examples/fm_radio.rs:84-87) fused in front, so HBM carries 2 instead of 8 bytes per input sample.  Fused
 * inside the TMA-staged kernel for real taps <= 64, decimation 5 or 10, n_in % 8 == 0 and a 16-byte aligned
 * input (there the span holds b - 127.5 exactly and the division by 127.5 sits in the taps: results equal to
 * convert-then-filter up to rounding, ~1e-7 relative); any other shape converts into an internal f32 scratch first
 * (bit-identical to convert-then-filter).  The carried state is ConvertNode's exact output either way. */
CB_API int cb_chain_run_u8(cb_chain *h, const uint8_t *in, size_t n_in, float *out, size_t out_cap_per_channel,
                           size_t *n_out_per_channel);
CB_API int cb_chain_run_u8_dev(cb_chain *h, const uint8_t *d_in, size_t n_in, float *d_out,
                               size_t out_cap_per_channel, size_t *n_out_per_channel, void *stream);
CB_API int cb_chain_run_dev(cb_chain *h, const float *d_in, size_t n_in, float *d_out,
                            size_t out_cap_per_channel, size_t *n_out_per_channel, void *stream);

/* ------------------------------------------------------------------ pulse-shaping taps (host side)
 * rrc_taps<T> (src/util/math.rs:221-280): root-raised-cosine impulse response
 * sampled at t_i = (i - (n_taps-1)/2) / sam_per_sym, T_sym = 1, evaluated in f64
 * with the reference's special cases (|t| < f64::EPSILON; |t -/+ 1/(4 beta)| <
 * f64::EPSILON) and no energy normalisation; imaginary parts are 0.
 * beta outside [0, 1] -> CB_ERR_INVALID_ARG (the reference's InvalidRolloffError).
 * taps: 2*n_taps floats (cb_rrc_taps: the f64 values cast to f32 like
 * T::from(f64)) or 2*n_taps doubles (cb_rrc_taps_f64).  Needs no device. */
CB_API int cb_rrc_taps(uint32_t n_taps, double sam_per_sym, double beta, float *taps);
CB_API int cb_rrc_taps_f64(uint32_t n_taps, double sam_per_sym, double beta, double *taps);

/* Stream argument of the *_dev entry points: a cudaStream_t, or NULL.  For entries that take a handle
 * NULL means the handle's own non-blocking stream; for the stateless entries below NULL is the legacy
 * default stream, which does NOT order against the handles' streams.  Pass one explicit stream when
 * chaining both kinds (as every device-resident example graph does). */

/* ------------------------------------------------------------------ bit-exact edges
 * Integer / index stages of the example graphs, device side, so whole example
 * chains can stay on the GPU.
 * cb_prn_bits: PrnGen::next_byte (src/prns.rs:64-71), `width` = register bits.
 * cb_bits_to_symbols: the example maps, mode 0 = BPSK b -> (2b-1) + 0j
 *   (examples/single_thread_bpsk.rs:29-32), mode 1 = QPSK bit pairs
 *   (examples/single_thread_qpsk.rs:29-36).
 * cb_quantize_i16: (scale * x) as i16, truncating and saturating
 *   (examples/single_thread_bpsk.rs:40-48). */
CB_API int cb_prn_bits(uint64_t poly_mask, uint64_t *state, unsigned width, size_t n, uint8_t *bits_host);
CB_API int cb_bits_to_symbols_dev(const uint8_t *d_bits, size_t nbits, int mode, float *d_sym,
                                  size_t *nsym, void *stream);
CB_API int cb_quantize_i16_dev(const float *d_in, size_t nfloats, float scale, int16_t *d_out, void *stream);
/* IQ edge formats.  cb_convert_u8: RTL-SDR bytes (u8 I, u8 Q) -> complex f32 by
 * (x as f32 - 127.5) / 127.5 (ConvertNode, examples/fm_radio.rs:84-87), exactly
 * rounded.  cb_convert_i16: the interleaved native-endian i16 IQ of
 * src/io/raw_iq.rs:20-140 -> scale * (x as f32) (scale = 1: the plain cast).
 * n_samples complex samples each; d_out receives 2*n_samples floats. */
/* ------------------------------------------------------------------ f64 estimators
 * The two feed-forward estimators of src/demodulation that call batch_fir (complex f64 samples = 2n interleaved
 * doubles).  Each call is one fused pass (filter, product, reduction) and returns its scalar on the host, so it
 * synchronises the stream it ran on.
 * d_samples of the _dev forms must be 16-byte aligned (read as pairs of doubles); other pointers return
 * CB_ERR_INVALID_ARG before any launch.
 * cb_freq_estimate: frequency_offset_estimate (src/demodulation/frequency_estimator.rs:27-42), radians/sample:
 *   arg(sum_{i<n-1} x[i+1] conj(x[i])); n < 2 gives 0.
 *   Accuracy: |est - arg S| <= asin(E / |S|) + 2^-49 (S the exact sum) whenever E < |S|, with
 *   E = sqrt(2) u64 D sum |x[i+1]| |x[i]|, D = m + ceil(P / 256) + 26, P = min(ceil(n / 2048), 1184) CTAs and
 *   m = ceil((n - 1) / (256 P)) terms per thread.  When E >= |S| the estimate is finite but carries no guarantee.
 *   A NaN sample gives NaN.
 * cb_timing_*: TimingEstimator::new / push (src/demodulation/timing_estimator.rs:43-58, 85-112), result in
 *   samples; alpha outside [0, 1] -> CB_ERR_INVALID_ARG (MathError::InvalidRolloffError); the internal filter
 *   length 2*n*d+1 is limited to 4097 (CB_ERR_UNSUPPORTED beyond).
 *   Accuracy: |est - est_exact| <= (n / 2 pi) (asin(E / |S|) + 2^-49) whenever E < |S|, S = sum_i qout_i dout_i exact
 *   (the reference's r_m = exp(-j fl(fl(-pi m) / n)) argument), E = u64 (sqrt(2) (ntaps4 + D) + 16) sum_i |dout_i| A_i,
 *   A_i = sum_k |q_k| |qin_{i-k}|, ntaps4 = the tap count rounded up to four, D = 4 ceil(T / P) + ceil(P / 256) + 26
 *   for T = ceil(len / 1024) tiles over P = min(T, 1184) CTAs.
 * cb_qfilt_taps_f64: qfilt_taps (src/util/math.rs:307-342); taps must hold n_taps + 1 doubles (an even n_taps is
 *   incremented by one); *n_out receives the count written. */
typedef struct cb_timing cb_timing;
CB_API int cb_qfilt_taps_f64(uint32_t n_taps, double alpha, uint32_t sam_per_sym, double *taps, uint32_t *n_out);
CB_API int cb_freq_estimate(const double *samples, size_t n, double *estimate);
CB_API int cb_freq_estimate_dev(const double *d_samples, size_t n, double *estimate, void *stream);
CB_API int cb_timing_create(uint32_t n, uint32_t d, double alpha, cb_timing **out);
CB_API int cb_timing_destroy(cb_timing *h);
CB_API int cb_timing_push(cb_timing *h, const double *samples, size_t n, double *estimate);
CB_API int cb_timing_push_dev(cb_timing *h, const double *d_samples, size_t n, double *estimate, void *stream);

/* ------------------------------------------------------------------ NCO
 * NcoNode::new(dphase, phase) / Nco::push (src/demodulation/nco.rs:41-49, 71-77, 112-127) over a batch of phase errors:
 *   phase_k = phase_{k-1} + dphase + perr[k]  (one conditional wrap when > 2 pi),  out[k] = exp(j * phase_k),
 * i.e. phase_k = phase_0 + (k+1)*dphase + sum_{i<=k} perr[i] (mod 2 pi): a prefix sum, evaluated as a device scan in
 * f64 with the ramp term reduced exactly; the wrap only picks the representative of the phase, never the output.
 * n doubles in -> n complex f64 (2n doubles) out; dphase wrapped into [0, 2 pi) like Nco::new; phase carried across
 * calls (cb_nco_get_phase returns it reduced to [0, 2 pi)).  At most 2^29 - 1 errors per call.
 * Accuracy, causal: output k depends on perr[0..k] only, and
 *   |out[k] - exp(j phi_k)| <= u64 (2 (|phase_0| + 2 pi (1 + calls_k + chunks_k)) + 16 S_k + 6),
 * phi_k the exact phase from the stream's start (or from the last cb_nco_set_phase, phase_0 its phase),
 * S_k = sum_{i<=k} |perr[i]|, calls_k = calls before the one holding k, chunks_k = (k within its call) / 2^21.
 * A NaN or infinite perr[j] makes out[j..] and the carried phase NaN, as in the reference recurrence; out[0..j-1]
 * keep the bound.  A huge perr[j] enters the bound of out[j..] only. */
typedef struct cb_nco cb_nco;
CB_API int cb_nco_create(double dphase, double phase, cb_nco **out);
CB_API int cb_nco_destroy(cb_nco *h);
CB_API int cb_nco_run(cb_nco *h, const double *perr, size_t n, double *out);
CB_API int cb_nco_run_dev(cb_nco *h, const double *d_perr, size_t n, double *d_out, void *stream);
CB_API int cb_nco_get_phase(cb_nco *h, double *phase, double *dphase);
CB_API int cb_nco_set_phase(cb_nco *h, double phase);

/* Real <-> complex glue of examples/fm_radio.rs, device side, so the whole shipped graph can stay on the GPU:
 * cb_real_to_complex: Convert2Node (fm_radio.rs:98-118), x -> Complex(x, 0); cb_complex_real: Convert3Node
 * (fm_radio.rs:122-142), z -> z.re.  n elements each. */
CB_API int cb_real_to_complex_dev(const float *d_in, size_t n, float *d_out, void *stream);
CB_API int cb_complex_real_dev(const float *d_in, size_t n, float *d_out, void *stream);
CB_API int cb_convert_u8_dev(const uint8_t *d_in, size_t n_samples, float *d_out, void *stream);
CB_API int cb_convert_i16_dev(const int16_t *d_in, size_t n_samples, float scale, float *d_out, void *stream);

/* ------------------------------------------------------------------ multi-GPU: ordered gather of segments
 * One process (or thread + cb_init) per GPU.  Channels, frames and overlap-save segments are computed without any
 * exchange (each rank passes the samples before its segment as the FIR's initial state, fir_node.rs:193-200); the
 * one collective is the optional gather of equal-length output segments back into one rank-ordered stream, an
 * ncclAllGather over NVLink.  NCCL is dlopen'ed on first use (libnccl.so.2, or COMMS_B200_NCCL_LIB), so the
 * library does not depend on it otherwise; CB_ERR_UNSUPPORTED when it cannot be loaded.
 * cb_comm_unique_id: rank 0 creates the 128-byte id and hands it to the other ranks by any host channel.
 * cb_gather_segments_dev: d_all receives nranks * n_samples complex samples, rank r's segment at r * n_samples. */
typedef struct cb_comm cb_comm;
CB_API int cb_comm_unique_id(void *id128);
CB_API int cb_comm_init(int nranks, int rank, const void *id128, cb_comm **out);
CB_API int cb_comm_destroy(cb_comm *c);
CB_API int cb_comm_rank(const cb_comm *c, int *rank, int *nranks);
/* Equal-length segments onto EVERY rank (ncclAllGather).  A collective: every rank must call it with the same
 * n_samples (0 everywhere is a no-op everywhere; one rank may not skip the call on its own). */
CB_API int cb_gather_segments_dev(cb_comm *c, const float *d_seg, size_t n_samples, float *d_all, void *stream);
/* Ordered gather of segments of ANY lengths onto ONE rank (what a single ordered output stream needs): counts[r]
 * elements of elem_bytes bytes from rank r land at d_all + sum_{q<r} counts[q] on `root`.  Every rank passes the
 * same counts[nranks] (the segment table is host knowledge, sharding.segment_bounds), so empty trailing segments are
 * skipped consistently and no rank blocks alone.  One grouped ncclSend/ncclRecv: the root's NVLink ingress carries
 * each remote byte once -- 1/nranks of the switch traffic of an all-gather.  d_all may be NULL off the root. */
CB_API int cb_gather_segments_to_root_dev(cb_comm *c, const void *d_seg, const size_t *counts, size_t elem_bytes,
                                          int root, void *d_all, void *stream);
/* The same ordered stream on every rank, segments of any lengths (one grouped broadcast per non-empty segment). */
CB_API int cb_allgather_segments_var_dev(cb_comm *c, const void *d_seg, const size_t *counts, size_t elem_bytes,
                                         void *d_all, void *stream);
/* Gather fused into the producing kernel: the root exports its gathered-stream buffer (64-byte CUDA IPC handle, passed
 * by any host channel; the pointer must be the base of a cb_buf_alloc_device / cudaMalloc allocation), the other
 * ranks map it and pass `mapped + byte offset of their segment` as d_out of cb_fir_run_dev / cb_chain_run_dev /
 * cb_fft_run_dev: the kernel's stores travel over NVLink / NVSwitch into the root's HBM tile by tile while the
 * filter runs; there is no second pass over the data and no collective call. */
CB_API int cb_peer_export(void *d_ptr, void *handle64);
CB_API int cb_peer_open(const void *handle64, void **d_mapped);
CB_API int cb_peer_close(void *d_mapped);

/* ------------------------------------------------------------------ synthetic input
 * splitmix64 counter generator shared with the oracle (oracle.c
 * orc_synth_uniform_f32): float i = top 24 bits of splitmix64(seed + i)
 * scaled to [-1, 1).  Fills n complex samples starting at complex index
 * `first`.  Used by tests and bench only. */
CB_API int cb_synth_uniform_dev(uint64_t seed, uint64_t first, size_t n, float *d_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* COMMS_B200_H */
