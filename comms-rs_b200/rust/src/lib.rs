//! GPU-backed drop-ins for the comms-rs nodes on the FIR / mixer / FFT hot path.
//!
//! Every struct keeps the reference's field spelling (`pub input: NodeReceiver<..>`,
//! `pub output: NodeSender<..>`; the derive macro classifies fields by that type text,
//! node_derive/src/lib.rs:240-250), constructor arguments and `run()` signature, so
//! `connect_nodes!` / `start_nodes!` / `Graph` work unchanged:
//!
//! ```ignore
//! use comms_b200::GpuBatchFirNode as BatchFirNode;   // instead of comms_rs::filter::fir_node::BatchFirNode
//! let mut filt = BatchFirNode::new(taps, None);
//! connect_nodes!(src, output, filt, input);
//! start_nodes!(src, filt);
//! ```
//!
//! Only `Complex<f32>` streams are accelerated (the element type of every BASELINE config).
#[macro_use]
extern crate comms_rs;

pub mod ffi;

use comms_rs::prelude::*;
use num::Complex;
use std::ffi::CStr;
use std::ptr;

type C32 = Complex<f32>;

/// cb_status -> NodeError (src/node/mod.rs:68-73): bad arguments / sizes are DataError,
/// anything else (CUDA failure, no device, OOM) stops the node for good.
fn check(status: i32) -> Result<(), NodeError> {
    match status {
        ffi::CB_OK => Ok(()),
        ffi::CB_ERR_INVALID_ARG | ffi::CB_ERR_SIZE => Err(NodeError::DataError),
        _ => {
            let msg = unsafe { CStr::from_ptr(ffi::cb_last_error()) };
            eprintln!("comms-b200: {}", msg.to_string_lossy());
            Err(NodeError::PermanentError)
        }
    }
}

fn as_f32(v: &[C32]) -> *const f32 { v.as_ptr() as *const f32 } // Complex<f32> is #[repr(C)] {re, im}

macro_rules! handle {
    ($name:ident, $raw:ty, $destroy:path) => {
        struct $name(*mut $raw);
        unsafe impl Send for $name {} // Node: Send; a handle is used by one thread at a time
        impl Drop for $name { fn drop(&mut self) { unsafe { $destroy(self.0); } } }
    };
}
handle!(Fir, ffi::cb_fir, ffi::cb_fir_destroy);
handle!(Mixer, ffi::cb_mixer, ffi::cb_mixer_destroy);
handle!(Fft, ffi::cb_fft, ffi::cb_fft_destroy);
handle!(Fm, ffi::cb_fm, ffi::cb_fm_destroy);

fn fir_new(taps: &[C32], state: Option<&[C32]>, decim: u32, interp: u32) -> Fir {
    let mut h = ptr::null_mut();
    let (sp, sn) = state.map_or((ptr::null(), 0), |s| (as_f32(s), s.len()));
    let st = unsafe { ffi::cb_fir_create(as_f32(taps), taps.len(), sp, sn, decim, interp, &mut h) };
    assert_eq!(st, ffi::CB_OK, "cb_fir_create failed (no CUDA device?)");
    Fir(h)
}

fn fir_run(h: &Fir, input: &[C32]) -> Result<Vec<C32>, NodeError> {
    let mut n_out = 0usize;
    check(unsafe { ffi::cb_fir_out_len(h.0, input.len(), &mut n_out) })?;
    let mut out: Vec<C32> = Vec::with_capacity(n_out);
    check(unsafe { ffi::cb_fir_run(h.0, as_f32(input), input.len(), out.as_mut_ptr() as *mut f32, n_out, &mut n_out) })?;
    unsafe { out.set_len(n_out) };
    Ok(out)
}

/// Drop-in for `util::math::rrc_taps::<f32>` (src/util/math.rs:221-280), evaluated by the library's
/// host entry so that the taps fed to the GPU filters are the reference's, bit for bit.
pub fn rrc_taps(n_taps: u32, sam_per_sym: f64, beta: f64) -> Result<Vec<C32>, comms_rs::util::MathError> {
    let mut taps: Vec<C32> = vec![Complex::new(0.0, 0.0); n_taps as usize];
    match unsafe { ffi::cb_rrc_taps(n_taps, sam_per_sym, beta, taps.as_mut_ptr() as *mut f32) } {
        ffi::CB_OK => Ok(taps),
        _ => Err(comms_rs::util::MathError::InvalidRolloffError),
    }
}

/// Drop-in for `BatchFirNode<f32>` (src/filter/fir_node.rs:146-221).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuBatchFirNode {
    pub input: NodeReceiver<Vec<C32>>,
    fir: Fir,
    pub output: NodeSender<Vec<C32>>,
}

impl GpuBatchFirNode {
    pub fn new(taps: Vec<C32>, state: Option<Vec<C32>>) -> Self {
        GpuBatchFirNode { fir: fir_new(&taps, state.as_deref(), 1, 1), input: Default::default(), output: Default::default() }
    }
    /// FIR with the neighbouring `UpsampleNode(interp)` / `DecimateNode(decim)` fused.
    pub fn with_resampling(taps: Vec<C32>, state: Option<Vec<C32>>, decim: u32, interp: u32) -> Self {
        GpuBatchFirNode { fir: fir_new(&taps, state.as_deref(), decim, interp), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[C32]) -> Result<Vec<C32>, NodeError> { fir_run(&self.fir, input) }
}

/// Drop-in for `FirNode<f32>` (src/filter/fir_node.rs:43-114): one sample per message.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuFirNode {
    pub input: NodeReceiver<C32>,
    fir: Fir,
    pub output: NodeSender<C32>,
}

impl GpuFirNode {
    pub fn new(taps: Vec<C32>, state: Option<Vec<C32>>) -> Self {
        GpuFirNode { fir: fir_new(&taps, state.as_deref(), 1, 1), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &C32) -> Result<C32, NodeError> {
        Ok(fir_run(&self.fir, std::slice::from_ref(input))?[0])
    }
}

/// Drop-in for `PulseNode<f32>` (src/pulse.rs:36-92): one symbol in, `sam_per_sym` samples out.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuPulseNode {
    pub input: NodeReceiver<C32>,
    fir: Fir,
    pub output: NodeSender<Vec<C32>>,
}

impl GpuPulseNode {
    pub fn new(taps: Vec<C32>, sam_per_sym: usize) -> Self {
        GpuPulseNode { fir: fir_new(&taps, None, 1, sam_per_sym as u32), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &C32) -> Result<Vec<C32>, NodeError> { fir_run(&self.fir, std::slice::from_ref(input)) }
}

/// Batched form of the pulse shaper: `Vec` of symbols in, `sam_per_sym` x as many samples out
/// (what UpsampleNode -> BatchFirNode does in examples/bpsk_mod.rs:153-155).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuBatchPulseNode {
    pub input: NodeReceiver<Vec<C32>>,
    fir: Fir,
    pub output: NodeSender<Vec<C32>>,
}

impl GpuBatchPulseNode {
    pub fn new(taps: Vec<C32>, sam_per_sym: usize) -> Self {
        GpuBatchPulseNode { fir: fir_new(&taps, None, 1, sam_per_sym as u32), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[C32]) -> Result<Vec<C32>, NodeError> { fir_run(&self.fir, input) }
}

type C64 = Complex<f64>;
handle!(FirF64, ffi::cb_fir_f64, ffi::cb_fir_f64_destroy);

fn as_f64(v: &[C64]) -> *const f64 { v.as_ptr() as *const f64 } // Complex<f64> is #[repr(C)] {re, im}

fn fir_f64_new(taps: &[C64], state: Option<&[C64]>, decim: u32, interp: u32) -> FirF64 {
    let mut h = ptr::null_mut();
    let (sp, sn) = state.map_or((ptr::null(), 0), |s| (as_f64(s), s.len()));
    let st = unsafe { ffi::cb_fir_f64_create(as_f64(taps), taps.len(), sp, sn, decim, interp, &mut h) };
    assert_eq!(st, ffi::CB_OK, "cb_fir_f64_create failed (non-finite tap, or no CUDA device?)");
    FirF64(h)
}

fn fir_f64_run(h: &FirF64, input: &[C64]) -> Result<Vec<C64>, NodeError> {
    let mut n_out = 0usize;
    check(unsafe { ffi::cb_fir_f64_out_len(h.0, input.len(), &mut n_out) })?;
    let mut out: Vec<C64> = Vec::with_capacity(n_out);
    check(unsafe { ffi::cb_fir_f64_run(h.0, as_f64(input), input.len(), out.as_mut_ptr() as *mut f64, n_out, &mut n_out) })?;
    unsafe { out.set_len(n_out) };
    Ok(out)
}

/// Drop-in for `BatchFirNode<f64>` (src/filter/fir_node.rs:146-221) over `Complex<f64>`.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuBatchFirNodeF64 {
    pub input: NodeReceiver<Vec<C64>>,
    fir: FirF64,
    pub output: NodeSender<Vec<C64>>,
}

impl GpuBatchFirNodeF64 {
    pub fn new(taps: Vec<C64>, state: Option<Vec<C64>>) -> Self {
        GpuBatchFirNodeF64 { fir: fir_f64_new(&taps, state.as_deref(), 1, 1), input: Default::default(), output: Default::default() }
    }
    /// FIR with the neighbouring `UpsampleNode(interp)` / `DecimateNode(decim)` fused.
    pub fn with_resampling(taps: Vec<C64>, state: Option<Vec<C64>>, decim: u32, interp: u32) -> Self {
        GpuBatchFirNodeF64 { fir: fir_f64_new(&taps, state.as_deref(), decim, interp), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[C64]) -> Result<Vec<C64>, NodeError> { fir_f64_run(&self.fir, input) }
}

/// Drop-in for `PulseNode<f64>` (src/pulse.rs:36-92): one symbol in, `sam_per_sym` samples out.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuPulseNodeF64 {
    pub input: NodeReceiver<C64>,
    fir: FirF64,
    pub output: NodeSender<Vec<C64>>,
}

impl GpuPulseNodeF64 {
    pub fn new(taps: Vec<C64>, sam_per_sym: usize) -> Self {
        GpuPulseNodeF64 { fir: fir_f64_new(&taps, None, 1, sam_per_sym as u32), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &C64) -> Result<Vec<C64>, NodeError> { fir_f64_run(&self.fir, std::slice::from_ref(input)) }
}

/// Drop-in for `DecimateNode<T>` (src/util/resample_node.rs:18-65) for plain-old-data `T`.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuDecimateNode<T>
where
    T: Copy + Send,
{
    pub input: NodeReceiver<Vec<T>>,
    dec_rate: usize,
    pub output: NodeSender<Vec<T>>,
}

impl<T: Copy + Send> GpuDecimateNode<T> {
    pub fn new(dec_rate: usize) -> Self { GpuDecimateNode { dec_rate, input: Default::default(), output: Default::default() } }
    pub fn run(&mut self, input: &[T]) -> Result<Vec<T>, NodeError> {
        let cap = if self.dec_rate <= 1 { input.len() } else { (input.len() + self.dec_rate - 1) / self.dec_rate };
        let mut out: Vec<T> = Vec::with_capacity(cap);
        let mut n = 0usize;
        check(unsafe { ffi::cb_decimate(input.as_ptr() as *const _, input.len(), std::mem::size_of::<T>(), self.dec_rate,
                                        out.as_mut_ptr() as *mut _, cap, &mut n) })?;
        unsafe { out.set_len(n) };
        Ok(out)
    }
}

/// Drop-in for `UpsampleNode<T>` (src/util/resample_node.rs:82-131); zero = all-zero bytes.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuUpsampleNode<T>
where
    T: Copy + Send,
{
    pub input: NodeReceiver<Vec<T>>,
    ups_rate: usize,
    pub output: NodeSender<Vec<T>>,
}

impl<T: Copy + Send> GpuUpsampleNode<T> {
    pub fn new(ups_rate: usize) -> Self { GpuUpsampleNode { ups_rate, input: Default::default(), output: Default::default() } }
    pub fn run(&mut self, input: &[T]) -> Result<Vec<T>, NodeError> {
        let cap = if self.ups_rate <= 1 { input.len() } else { input.len() * self.ups_rate };
        let mut out: Vec<T> = Vec::with_capacity(cap);
        let mut n = 0usize;
        check(unsafe { ffi::cb_upsample(input.as_ptr() as *const _, input.len(), std::mem::size_of::<T>(), self.ups_rate,
                                        out.as_mut_ptr() as *mut _, cap, &mut n) })?;
        unsafe { out.set_len(n) };
        Ok(out)
    }
}

/// Drop-in for `MixerNode<f32>` (src/mixer.rs:91-148); note `new(dphase, phase)`.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuMixerNode {
    pub input: NodeReceiver<C32>,
    mixer: Mixer,
    pub output: NodeSender<C32>,
}

fn mixer_new(dphase: f64, phase: Option<f64>) -> Mixer {
    let mut h = ptr::null_mut();
    let st = unsafe { ffi::cb_mixer_create(dphase, phase.unwrap_or(0.0), &mut h) };
    assert_eq!(st, ffi::CB_OK, "cb_mixer_create failed");
    Mixer(h)
}

impl GpuMixerNode {
    pub fn new(dphase: f64, phase: Option<f64>) -> Self {
        GpuMixerNode { mixer: mixer_new(dphase, phase), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &C32) -> Result<C32, NodeError> {
        let mut out = C32::new(0.0, 0.0);
        check(unsafe { ffi::cb_mixer_run(self.mixer.0, input as *const C32 as *const f32, 1, &mut out as *mut C32 as *mut f32) })?;
        Ok(out)
    }
}

/// Batched mixer (no counterpart node in the reference, which mixes one sample per message).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuBatchMixerNode {
    pub input: NodeReceiver<Vec<C32>>,
    mixer: Mixer,
    pub output: NodeSender<Vec<C32>>,
}

impl GpuBatchMixerNode {
    pub fn new(dphase: f64, phase: Option<f64>) -> Self {
        GpuBatchMixerNode { mixer: mixer_new(dphase, phase), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[C32]) -> Result<Vec<C32>, NodeError> {
        let mut out: Vec<C32> = Vec::with_capacity(input.len());
        check(unsafe { ffi::cb_mixer_run(self.mixer.0, as_f32(input), input.len(), out.as_mut_ptr() as *mut f32) })?;
        unsafe { out.set_len(input.len()) };
        Ok(out)
    }
}

/// Drop-in for `NcoNode` (src/demodulation/nco.rs:82-133): one phase error in, one `Complex<f64>` out.
#[derive(Node)]
pub struct GpuNcoNode {
    pub input: NodeReceiver<f64>,
    nco: Nco,
    pub output: NodeSender<Complex<f64>>,
}

struct Nco(*mut ffi::cb_nco);
unsafe impl Send for Nco {}
impl Drop for Nco {
    fn drop(&mut self) {
        unsafe { ffi::cb_nco_destroy(self.0) };
    }
}

fn nco_new(dphase: f64, phase: Option<f64>) -> Nco {
    let mut h = ptr::null_mut();
    let st = unsafe { ffi::cb_nco_create(dphase, phase.unwrap_or(0.0), &mut h) };
    assert_eq!(st, ffi::CB_OK, "cb_nco_create failed");
    Nco(h)
}

impl GpuNcoNode {
    pub fn new(dphase: f64, phase: Option<f64>) -> Self {
        GpuNcoNode { nco: nco_new(dphase, phase), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: f64) -> Result<Complex<f64>, NodeError> {
        let mut out = Complex::new(0.0f64, 0.0f64);
        check(unsafe { ffi::cb_nco_run(self.nco.0, &input, 1, &mut out as *mut Complex<f64> as *mut f64) })?;
        Ok(out)
    }
}

/// Batching shim: a vector of phase errors per message, `Nco::push` applied in order on the device (one scan).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuNcoBatchNode {
    pub input: NodeReceiver<Vec<f64>>,
    nco: Nco,
    pub output: NodeSender<Vec<Complex<f64>>>,
}

impl GpuNcoBatchNode {
    pub fn new(dphase: f64, phase: Option<f64>) -> Self {
        GpuNcoBatchNode { nco: nco_new(dphase, phase), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[f64]) -> Result<Vec<Complex<f64>>, NodeError> {
        let mut out: Vec<Complex<f64>> = Vec::with_capacity(input.len());
        check(unsafe { ffi::cb_nco_run(self.nco.0, input.as_ptr(), input.len(), out.as_mut_ptr() as *mut f64) })?;
        unsafe { out.set_len(input.len()) };
        Ok(out)
    }
}

/// Drop-in for `FFTBatchNode<f32>` (src/fft/fft_node.rs:26-84).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuFFTBatchNode {
    pub input: NodeReceiver<Vec<C32>>,
    fft: Fft,
    pub output: NodeSender<Vec<C32>>,
}

fn fft_new(fft_size: usize, ifft: bool) -> Fft {
    let mut h = ptr::null_mut();
    let st = unsafe { ffi::cb_fft_create(fft_size, ifft as i32, &mut h) };
    assert_eq!(st, ffi::CB_OK, "cb_fft_create failed");
    Fft(h)
}

impl GpuFFTBatchNode {
    pub fn new(fft_size: usize, ifft: bool) -> Self {
        GpuFFTBatchNode { fft: fft_new(fft_size, ifft), input: Default::default(), output: Default::default() }
    }
    /// A length that is not a multiple of fft_size is a DataError (rustfft would panic the node thread).
    pub fn run(&mut self, data: &[C32]) -> Result<Vec<C32>, NodeError> {
        let mut out: Vec<C32> = Vec::with_capacity(data.len());
        check(unsafe { ffi::cb_fft_run(self.fft.0, as_f32(data), data.len(), out.as_mut_ptr() as *mut f32) })?;
        unsafe { out.set_len(data.len()) };
        Ok(out)
    }
}

/// Drop-in for `FFTSampleNode<f32>` (src/fft/fft_node.rs:101-168).
#[derive(Node)]
#[aggregate]
#[pass_by_ref]
pub struct GpuFFTSampleNode {
    pub input: NodeReceiver<C32>,
    fft: Fft,
    fft_size: usize,
    samples: Vec<C32>,
    pub output: NodeSender<Vec<C32>>,
}

impl GpuFFTSampleNode {
    pub fn new(fft_size: usize, ifft: bool) -> Self {
        GpuFFTSampleNode { fft: fft_new(fft_size, ifft), fft_size, samples: Vec::with_capacity(fft_size),
                           input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &C32) -> Result<Option<Vec<C32>>, NodeError> {
        self.samples.push(*input);
        if self.samples.len() == self.fft_size {
            let mut out: Vec<C32> = Vec::with_capacity(self.fft_size);
            check(unsafe { ffi::cb_fft_run(self.fft.0, as_f32(&self.samples), self.fft_size, out.as_mut_ptr() as *mut f32) })?;
            unsafe { out.set_len(self.fft_size) };
            self.samples.clear();
            Ok(Some(out))
        } else {
            Ok(None)
        }
    }
}

handle!(FftF64, ffi::cb_fft_f64, ffi::cb_fft_f64_destroy);

fn fft_f64_new(fft_size: usize, ifft: bool) -> FftF64 {
    let mut h = ptr::null_mut();
    let st = unsafe { ffi::cb_fft_f64_create(fft_size, ifft as i32, &mut h) };
    assert_eq!(st, ffi::CB_OK, "cb_fft_f64_create failed");
    FftF64(h)
}

fn fft_f64_run(h: &FftF64, data: &[C64]) -> Result<Vec<C64>, NodeError> {
    let mut out: Vec<C64> = Vec::with_capacity(data.len());
    check(unsafe { ffi::cb_fft_f64_run(h.0, as_f64(data), data.len(), out.as_mut_ptr() as *mut f64) })?;
    unsafe { out.set_len(data.len()) };
    Ok(out)
}

/// Drop-in for `FFTBatchNode<f64>` (src/fft/fft_node.rs:26-84) over `Complex<f64>`: the reference runs every
/// transform in f64 (src/fft/mod.rs:73-96), and so does `cb_fft_f64`.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuFFTBatchNodeF64 {
    pub input: NodeReceiver<Vec<C64>>,
    fft: FftF64,
    pub output: NodeSender<Vec<C64>>,
}

impl GpuFFTBatchNodeF64 {
    pub fn new(fft_size: usize, ifft: bool) -> Self {
        GpuFFTBatchNodeF64 { fft: fft_f64_new(fft_size, ifft), input: Default::default(), output: Default::default() }
    }
    /// A length that is not a multiple of fft_size is a DataError (rustfft would panic the node thread).
    pub fn run(&mut self, data: &[C64]) -> Result<Vec<C64>, NodeError> { fft_f64_run(&self.fft, data) }
}

/// Drop-in for `FFTSampleNode<f64>` (src/fft/fft_node.rs:101-168) over `Complex<f64>`.
#[derive(Node)]
#[aggregate]
#[pass_by_ref]
pub struct GpuFFTSampleNodeF64 {
    pub input: NodeReceiver<C64>,
    fft: FftF64,
    fft_size: usize,
    samples: Vec<C64>,
    pub output: NodeSender<Vec<C64>>,
}

impl GpuFFTSampleNodeF64 {
    pub fn new(fft_size: usize, ifft: bool) -> Self {
        GpuFFTSampleNodeF64 { fft: fft_f64_new(fft_size, ifft), fft_size, samples: Vec::with_capacity(fft_size),
                              input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &C64) -> Result<Option<Vec<C64>>, NodeError> {
        self.samples.push(*input);
        if self.samples.len() == self.fft_size {
            let out = fft_f64_run(&self.fft, &self.samples)?;
            self.samples.clear();
            Ok(Some(out))
        } else {
            Ok(None)
        }
    }
}

/// Drop-in for `FMDemodNode<f32>` (src/modulation/analog_node.rs:18-52).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuFMDemodNode {
    pub input: NodeReceiver<Vec<C32>>,
    fm: Fm,
    pub output: NodeSender<Vec<f32>>,
}

impl GpuFMDemodNode {
    pub fn new() -> Self {
        let mut h = ptr::null_mut();
        let st = unsafe { ffi::cb_fm_create(&mut h) };
        assert_eq!(st, ffi::CB_OK, "cb_fm_create failed");
        GpuFMDemodNode { fm: Fm(h), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, samples: &[C32]) -> Result<Vec<f32>, NodeError> {
        let mut out: Vec<f32> = Vec::with_capacity(samples.len());
        check(unsafe { ffi::cb_fm_run(self.fm.0, as_f32(samples), samples.len(), out.as_mut_ptr()) })?;
        unsafe { out.set_len(samples.len()) };
        Ok(out)
    }
}

/// What crosses a channel between two adjacent GPU nodes instead of a `Vec`: a ref-counted
/// device (or pinned-host) buffer.  `Clone` is a refcount bump -- the derive macro clones the
/// result once per downstream edge (node_derive/src/lib.rs:156) -- and `Drop` releases it.
pub struct DeviceBuf { raw: *mut ffi::cb_buf, pub len: usize }
unsafe impl Send for DeviceBuf {}
impl Clone for DeviceBuf {
    fn clone(&self) -> Self { unsafe { ffi::cb_buf_retain(self.raw) }; DeviceBuf { raw: self.raw, len: self.len } }
}
impl Drop for DeviceBuf { fn drop(&mut self) { unsafe { ffi::cb_buf_release(self.raw) }; } }
impl DeviceBuf {
    pub fn device(samples: usize) -> Result<Self, NodeError> {
        let mut raw = ptr::null_mut();
        check(unsafe { ffi::cb_buf_alloc_device(samples * 8, &mut raw) })?;
        Ok(DeviceBuf { raw, len: samples })
    }
    pub fn ptr(&self) -> *mut f32 { unsafe { ffi::cb_buf_ptr(self.raw) as *mut f32 } }
}

/// Device-resident FIR node: `DeviceBuf` in, `DeviceBuf` out, no host staging; used between
/// GPU nodes (e.g. mixer -> FIR -> FFT) so only graph edges touch PCIe.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuBatchFirDevNode {
    pub input: NodeReceiver<DeviceBuf>,
    fir: Fir,
    pub output: NodeSender<DeviceBuf>,
}

impl GpuBatchFirDevNode {
    pub fn new(taps: Vec<C32>, state: Option<Vec<C32>>) -> Self {
        GpuBatchFirDevNode { fir: fir_new(&taps, state.as_deref(), 1, 1), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &DeviceBuf) -> Result<DeviceBuf, NodeError> {
        let mut n_out = 0usize;
        check(unsafe { ffi::cb_fir_out_len(self.fir.0, input.len, &mut n_out) })?;
        let out = DeviceBuf::device(n_out)?;
        let stream = unsafe { ffi::cb_fir_stream(self.fir.0) };
        check(unsafe { ffi::cb_buf_wait_ready(input.raw, stream) })?; // producer's stream -> ours, no host sync
        check(unsafe { ffi::cb_fir_run_dev(self.fir.0, input.ptr(), input.len, out.ptr(), n_out, &mut n_out, stream) })?;
        // the pool hands `input`'s block to its next owner only after this launch has read it
        check(unsafe { ffi::cb_buf_record_done(input.raw, stream) })?;
        check(unsafe { ffi::cb_buf_record_ready(out.raw, stream) })?;
        Ok(out)
    }
}

/// Graph edge host -> device: a `Vec` in, a pooled `DeviceBuf` out.  This is where pool buffers START in a graph, so it
/// is also where the back-pressure gate sits: `cb_pool_throttle` blocks while more than the configured high-water mark
/// of device / pinned messages is in flight (comms-rs channels are unbounded, src/node/mod.rs:152).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuUploadNode {
    pub input: NodeReceiver<Vec<C32>>,
    stream: Stream,
    pub output: NodeSender<DeviceBuf>,
}

struct Stream(*mut ffi::cb_stream);
unsafe impl Send for Stream {}
impl Drop for Stream {
    fn drop(&mut self) {
        unsafe { ffi::cb_stream_destroy(self.0) };
    }
}

impl GpuUploadNode {
    pub fn new() -> Self {
        let mut s = ptr::null_mut();
        let st = unsafe { ffi::cb_stream_create(&mut s) };
        assert_eq!(st, ffi::CB_OK, "cb_stream_create failed");
        GpuUploadNode { stream: Stream(s), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[C32]) -> Result<DeviceBuf, NodeError> {
        check(unsafe { ffi::cb_pool_throttle(0) })?;
        let out = DeviceBuf::device(input.len())?;
        let s = unsafe { ffi::cb_stream_handle(self.stream.0) };
        check(unsafe { ffi::cb_copy_h2d_async(out.ptr() as *mut _, input.as_ptr() as *const _, input.len() * 8, s) })?;
        // `input` is borrowed for this call only: the copy must have left it before run() returns
        check(unsafe { ffi::cb_stream_sync(self.stream.0) })?;
        check(unsafe { ffi::cb_buf_record_ready(out.raw, s) })?;
        Ok(out)
    }
}

/// Graph edge device -> host: a `DeviceBuf` in, a `Vec` out.
#[derive(Node)]
#[pass_by_ref]
pub struct GpuDownloadNode {
    pub input: NodeReceiver<DeviceBuf>,
    stream: Stream,
    pub output: NodeSender<Vec<C32>>,
}

impl GpuDownloadNode {
    pub fn new() -> Self {
        let mut s = ptr::null_mut();
        let st = unsafe { ffi::cb_stream_create(&mut s) };
        assert_eq!(st, ffi::CB_OK, "cb_stream_create failed");
        GpuDownloadNode { stream: Stream(s), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &DeviceBuf) -> Result<Vec<C32>, NodeError> {
        let mut out: Vec<C32> = Vec::with_capacity(input.len);
        let s = unsafe { ffi::cb_stream_handle(self.stream.0) };
        check(unsafe { ffi::cb_buf_wait_ready(input.raw, s) })?;
        check(unsafe { ffi::cb_copy_d2h_async(out.as_mut_ptr() as *mut _, input.ptr() as *const _, input.len * 8, s) })?;
        check(unsafe { ffi::cb_stream_sync(self.stream.0) })?;
        unsafe { out.set_len(input.len) };
        Ok(out)
    }
}

/// The second stage of `examples/fm_radio.rs` (`Convert2Node -> filt2 -> Convert3Node -> dec2`, :98-164) as one node:
/// real samples in, the real parts of the filtered and decimated stream out.  In the example it replaces the four
/// nodes between `fm` and `audio`; the ports keep the types of the outer two (`Vec<f32>` in, `Vec<f32>` out).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuRealFirDecimNode {
    pub input: NodeReceiver<Vec<f32>>,
    fir: Fir,
    pub output: NodeSender<Vec<f32>>,
}

impl GpuRealFirDecimNode {
    pub fn new(taps: Vec<C32>, state: Option<Vec<C32>>, dec_rate: u32) -> Self {
        GpuRealFirDecimNode { fir: fir_new(&taps, state.as_deref(), dec_rate.max(1), 1), input: Default::default(), output: Default::default() }
    }
    pub fn run(&mut self, input: &[f32]) -> Result<Vec<f32>, NodeError> {
        let mut n_out = 0usize;
        check(unsafe { ffi::cb_fir_out_len(self.fir.0, input.len(), &mut n_out) })?;
        let mut out: Vec<f32> = Vec::with_capacity(n_out);
        check(unsafe { ffi::cb_fir_run_real(self.fir.0, input.as_ptr(), input.len(), out.as_mut_ptr(), n_out, &mut n_out) })?;
        unsafe { out.set_len(n_out) };
        Ok(out)
    }
}

handle!(Timing, ffi::cb_timing, ffi::cb_timing_destroy);

/// Drop-in for `TimingEstimatorNode` (src/demodulation/timing_estimator.rs:116-137).
#[derive(Node)]
#[pass_by_ref]
pub struct GpuTimingEstimatorNode {
    pub input: NodeReceiver<Vec<num::Complex<f64>>>,
    est: Timing,
    pub output: NodeSender<f64>,
}

impl GpuTimingEstimatorNode {
    pub fn new(n: u32, d: u32, alpha: f64) -> Result<Self, comms_rs::util::MathError> {
        let mut h = ptr::null_mut();
        let st = unsafe { ffi::cb_timing_create(n, d, alpha, &mut h) };
        if st == ffi::CB_ERR_INVALID_ARG && !(0.0..=1.0).contains(&alpha) {
            return Err(comms_rs::util::MathError::InvalidRolloffError);
        }
        assert_eq!(st, ffi::CB_OK, "cb_timing_create failed");
        Ok(GpuTimingEstimatorNode { est: Timing(h), input: Default::default(), output: Default::default() })
    }
    pub fn run(&mut self, input: &[num::Complex<f64>]) -> Result<f64, NodeError> {
        let mut est = 0.0f64;
        check(unsafe { ffi::cb_timing_push(self.est.0, input.as_ptr() as *const f64, input.len(), &mut est) })?;
        Ok(est)
    }
}

/// Drop-in for `frequency_offset_estimate` (src/demodulation/frequency_estimator.rs:27-42).
pub fn frequency_offset_estimate(samples: &[num::Complex<f64>]) -> Result<f64, NodeError> {
    let mut est = 0.0f64;
    check(unsafe { ffi::cb_freq_estimate(samples.as_ptr() as *const f64, samples.len(), &mut est) })?;
    Ok(est)
}
