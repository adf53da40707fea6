// comms_b200_nodes.hpp -- C++ host-side mirror of the comms-rs node interface for the hot path,
// above the C ABI (include/comms_b200.h).  The reference is compiled Rust and this image has no
// rustc, so this header plays the role of the Rust shim (comms-rs_b200/rust/) in tests: same node
// names, constructor arguments, ports (`input` / `output`), run() meaning and error behaviour.
//
//   trait Node { start(); call() -> Result<(), NodeError>; is_connected() }   src/node/mod.rs:94-98
//   NodeReceiver<T> = Option<Receiver<T>>, NodeSender<T> = Vec<(Sender<T>, Option<T>)>
//                                                                              src/prelude.rs:9-10
//   call(): recv every input (Err -> DataEnd, unconnected -> PermanentError), run(), send a clone
//           to every output edge (Err -> CommError)               node_derive/src/lib.rs:199-211
//   start(): loop { if call().is_err() break }                    node_derive/src/lib.rs:181-197
//   connect_nodes!(a, output, b, input)                           src/node/mod.rs:150-156
//   start_nodes!(a, b, ...): one OS thread per node               src/node/mod.rs:276-284
#pragma once
#include <complex>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/comms_b200.h"

namespace comms_b200 {

using c32 = std::complex<float>;  // layout-compatible with num::Complex<f32> {re, im}

enum class NodeError { DataError, PermanentError, DataEnd, CommError };  // src/node/mod.rs:68-73

template <class T>
struct Result {
    std::optional<T> ok;
    NodeError err{};
    static Result Ok(T v) { Result r; r.ok = std::move(v); return r; }
    static Result Err(NodeError e) { Result r; r.err = e; return r; }
    bool is_ok() const { return ok.has_value(); }
};

inline NodeError map_status(int st)  // the shim's cb_status -> NodeError rule
{
    return (st == CB_ERR_INVALID_ARG || st == CB_ERR_SIZE) ? NodeError::DataError : NodeError::PermanentError;
}

// ---- crossbeam-like unbounded channel: recv() fails once every Sender is gone and the queue is empty
template <class T>
struct Chan {
    std::mutex m;
    std::condition_variable cv;
    std::deque<T> q;
    int senders = 0;
    bool receiver_alive = true;
};
template <class T>
class Sender {
    std::shared_ptr<Chan<T>> c_;
public:
    explicit Sender(std::shared_ptr<Chan<T>> c) : c_(std::move(c)) { std::lock_guard<std::mutex> l(c_->m); ++c_->senders; }
    Sender(const Sender &o) : c_(o.c_) { std::lock_guard<std::mutex> l(c_->m); ++c_->senders; }
    Sender(Sender &&o) noexcept : c_(std::move(o.c_)) {}
    Sender &operator=(const Sender &) = delete;
    ~Sender()
    {
        if (!c_) return;
        { std::lock_guard<std::mutex> l(c_->m); --c_->senders; }
        c_->cv.notify_all();
    }
    bool send(T v)
    {
        { std::lock_guard<std::mutex> l(c_->m); if (!c_->receiver_alive) return false; c_->q.push_back(std::move(v)); }
        c_->cv.notify_one();
        return true;
    }
};
template <class T>
class Receiver {
    std::shared_ptr<Chan<T>> c_;
public:
    explicit Receiver(std::shared_ptr<Chan<T>> c) : c_(std::move(c)) {}
    Receiver(Receiver &&) noexcept = default;
    Receiver &operator=(Receiver &&) noexcept = default;
    ~Receiver() { if (c_) { std::lock_guard<std::mutex> l(c_->m); c_->receiver_alive = false; } }
    std::optional<T> recv()
    {
        std::unique_lock<std::mutex> l(c_->m);
        c_->cv.wait(l, [&] { return !c_->q.empty() || c_->senders == 0; });
        if (c_->q.empty()) return std::nullopt;
        T v = std::move(c_->q.front());
        c_->q.pop_front();
        return v;
    }
};
template <class T> using NodeReceiver = std::optional<Receiver<T>>;
template <class T> using NodeSender = std::vector<Sender<T>>;

struct Node {
    virtual ~Node() = default;
    virtual Result<bool> call() = 0;
    virtual bool is_connected() const = 0;
    void start() { while (call().is_ok()) {} }
};

// The derived impl for a one-input one-output node (pass_by_ref), optional aggregate semantics.
template <class Derived, class In, class Out, bool Aggregate = false>
struct Node1 : Node {
    NodeReceiver<In> input;
    NodeSender<Out> output;
    bool is_connected() const override { return input.has_value(); }
    Result<bool> call() override
    {
        if (!input) return Result<bool>::Err(NodeError::PermanentError);
        auto msg = input->recv();
        if (!msg) { output.clear(); return Result<bool>::Err(NodeError::DataEnd); }
        if constexpr (Aggregate) {
            auto r = static_cast<Derived *>(this)->run(*msg);
            if (!r.is_ok()) { output.clear(); return Result<bool>::Err(r.err); }
            if (r.ok->has_value())
                for (auto &s : output) if (!s.send(**r.ok)) return Result<bool>::Err(NodeError::CommError);
        } else {
            auto r = static_cast<Derived *>(this)->run(*msg);
            if (!r.is_ok()) { output.clear(); return Result<bool>::Err(r.err); }  // node stops; senders drop
            for (auto &s : output) if (!s.send(*r.ok)) return Result<bool>::Err(NodeError::CommError);
        }
        return Result<bool>::Ok(true);
    }
};

template <class A, class B>
void connect_nodes(A &a, B &b)  // connect_nodes!(a, output, b, input)
{
    using Msg = typename decltype(std::declval<decltype(b.input)>()->recv())::value_type;
    auto ch = std::make_shared<Chan<Msg>>();
    a.output.emplace_back(ch);
    b.input.emplace(ch);
}

template <class... N>
std::vector<std::thread> start_nodes(N &...nodes)  // start_nodes!: a thread per node
{
    std::vector<std::thread> th;
    (th.emplace_back([&nodes] { nodes.start(); nodes.output.clear(); }), ...);
    return th;
}

// ------------------------------------------------------------------ GPU nodes
class FirHandle {
protected:
    cb_fir *h_ = nullptr;
public:
    FirHandle(const std::vector<c32> &taps, const std::vector<c32> *state, uint32_t decim, uint32_t interp)
    {
        int st = cb_fir_create(reinterpret_cast<const float *>(taps.data()), taps.size(),
                               state ? reinterpret_cast<const float *>(state->data()) : nullptr,
                               state ? state->size() : 0, decim, interp, &h_);
        if (st) throw std::runtime_error(std::string("cb_fir_create: ") + cb_last_error());
    }
    FirHandle(const FirHandle &) = delete;
    ~FirHandle() { cb_fir_destroy(h_); }
    Result<std::vector<c32>> filter(const c32 *in, size_t n)
    {
        size_t no = 0;
        cb_fir_out_len(h_, n, &no);
        std::vector<c32> out(no);
        int st = cb_fir_run(h_, reinterpret_cast<const float *>(in), n, reinterpret_cast<float *>(out.data()), no, &no);
        if (st) return Result<std::vector<c32>>::Err(map_status(st));
        out.resize(no);
        return Result<std::vector<c32>>::Ok(std::move(out));
    }
    std::vector<c32> state()
    {
        size_t n = 0;
        cb_fir_state_len(h_, &n);
        std::vector<c32> s(n);
        cb_fir_get_state(h_, reinterpret_cast<float *>(s.data()), n);
        return s;
    }
};

// BatchFirNode::new(taps, state) / run(&[Complex<T>])      src/filter/fir_node.rs:193-220
struct BatchFirNode : Node1<BatchFirNode, std::vector<c32>, std::vector<c32>>, FirHandle {
    BatchFirNode(const std::vector<c32> &taps, const std::vector<c32> *state = nullptr, uint32_t decim = 1, uint32_t interp = 1)
        : FirHandle(taps, state, decim, interp) {}
    Result<std::vector<c32>> run(const std::vector<c32> &in) { return filter(in.data(), in.size()); }
};

// FirNode: one sample per message                            src/filter/fir_node.rs:43-114
struct FirNode : Node1<FirNode, c32, c32>, FirHandle {
    FirNode(const std::vector<c32> &taps, const std::vector<c32> *state = nullptr) : FirHandle(taps, state, 1, 1) {}
    Result<c32> run(const c32 &in)
    {
        auto r = filter(&in, 1);
        return r.is_ok() ? Result<c32>::Ok((*r.ok)[0]) : Result<c32>::Err(r.err);
    }
};

// PulseNode::new(taps, sam_per_sym) / run(&Complex<T>) -> Vec  src/pulse.rs:71-92
struct PulseNode : Node1<PulseNode, c32, std::vector<c32>>, FirHandle {
    PulseNode(const std::vector<c32> &taps, size_t sam_per_sym) : FirHandle(taps, nullptr, 1, (uint32_t)sam_per_sym) {}
    Result<std::vector<c32>> run(const c32 &sym) { return filter(&sym, 1); }
};

// DecimateNode / UpsampleNode                                 src/util/resample_node.rs:18-131
template <class T>
struct DecimateNode : Node1<DecimateNode<T>, std::vector<T>, std::vector<T>> {
    size_t dec_rate;
    explicit DecimateNode(size_t r) : dec_rate(r) {}
    Result<std::vector<T>> run(const std::vector<T> &in)
    {
        size_t cap = dec_rate <= 1 ? in.size() : (in.size() + dec_rate - 1) / dec_rate, n = 0;
        std::vector<T> out(cap);
        int st = cb_decimate(in.data(), in.size(), sizeof(T), dec_rate, out.data(), cap, &n);
        if (st) return Result<std::vector<T>>::Err(map_status(st));
        out.resize(n);
        return Result<std::vector<T>>::Ok(std::move(out));
    }
};
template <class T>
struct UpsampleNode : Node1<UpsampleNode<T>, std::vector<T>, std::vector<T>> {
    size_t ups_rate;
    explicit UpsampleNode(size_t r) : ups_rate(r) {}
    Result<std::vector<T>> run(const std::vector<T> &in)
    {
        size_t cap = ups_rate <= 1 ? in.size() : in.size() * ups_rate, n = 0;
        std::vector<T> out(cap);
        int st = cb_upsample(in.data(), in.size(), sizeof(T), ups_rate, out.data(), cap, &n);
        if (st) return Result<std::vector<T>>::Err(map_status(st));
        out.resize(n);
        return Result<std::vector<T>>::Ok(std::move(out));
    }
};

// MixerNode::new(dphase, phase) / run(&Complex<T>)            src/mixer.rs:128-147
struct MixerNode : Node1<MixerNode, c32, c32> {
    cb_mixer *h_ = nullptr;
    explicit MixerNode(double dphase, std::optional<double> phase = std::nullopt)
    {
        if (cb_mixer_create(dphase, phase.value_or(0.0), &h_)) throw std::runtime_error(cb_last_error());
    }
    ~MixerNode() { cb_mixer_destroy(h_); }
    Result<c32> run(const c32 &in)
    {
        c32 out;
        int st = cb_mixer_run(h_, reinterpret_cast<const float *>(&in), 1, reinterpret_cast<float *>(&out));
        return st ? Result<c32>::Err(map_status(st)) : Result<c32>::Ok(out);
    }
};

// NcoNode::new(dphase, phase) / run(f64) -> Complex<f64>          src/demodulation/nco.rs:112-133
struct c64 {
    double re, im;
};
struct NcoNode : Node1<NcoNode, double, c64> {
    cb_nco *h_ = nullptr;
    explicit NcoNode(double dphase, std::optional<double> phase = std::nullopt)
    {
        if (cb_nco_create(dphase, phase.value_or(0.0), &h_)) throw std::runtime_error(cb_last_error());
    }
    ~NcoNode() { cb_nco_destroy(h_); }
    Result<c64> run(const double &perr)
    {
        c64 out;
        int st = cb_nco_run(h_, &perr, 1, reinterpret_cast<double *>(&out));
        return st ? Result<c64>::Err(map_status(st)) : Result<c64>::Ok(out);
    }
};

// Batching shim in front of GPU nodes: a vector of phase errors per message, the recurrence applied in order
struct NcoBatchNode : Node1<NcoBatchNode, std::vector<double>, std::vector<c64>> {
    cb_nco *h_ = nullptr;
    explicit NcoBatchNode(double dphase, std::optional<double> phase = std::nullopt)
    {
        if (cb_nco_create(dphase, phase.value_or(0.0), &h_)) throw std::runtime_error(cb_last_error());
    }
    ~NcoBatchNode() { cb_nco_destroy(h_); }
    Result<std::vector<c64>> run(const std::vector<double> &perr)
    {
        std::vector<c64> out(perr.size());
        int st = cb_nco_run(h_, perr.data(), perr.size(), reinterpret_cast<double *>(out.data()));
        return st ? Result<std::vector<c64>>::Err(map_status(st)) : Result<std::vector<c64>>::Ok(std::move(out));
    }
};

// The FIR over Complex<f64> (cb_fir_f64): same constructor arguments and run() meaning as the f32 nodes
class FirF64Handle {
protected:
    cb_fir_f64 *h_ = nullptr;
public:
    FirF64Handle(const std::vector<c64> &taps, const std::vector<c64> *state, uint32_t decim, uint32_t interp)
    {
        int st = cb_fir_f64_create(reinterpret_cast<const double *>(taps.data()), taps.size(),
                                   state ? reinterpret_cast<const double *>(state->data()) : nullptr,
                                   state ? state->size() : 0, decim, interp, &h_);
        if (st) throw std::runtime_error(std::string("cb_fir_f64_create: ") + cb_last_error());
    }
    FirF64Handle(const FirF64Handle &) = delete;
    ~FirF64Handle() { cb_fir_f64_destroy(h_); }
    Result<std::vector<c64>> filter(const c64 *in, size_t n)
    {
        size_t no = 0;
        cb_fir_f64_out_len(h_, n, &no);
        std::vector<c64> out(no);
        int st = cb_fir_f64_run(h_, reinterpret_cast<const double *>(in), n, reinterpret_cast<double *>(out.data()), no, &no);
        if (st) return Result<std::vector<c64>>::Err(map_status(st));
        out.resize(no);
        return Result<std::vector<c64>>::Ok(std::move(out));
    }
    std::vector<c64> state()
    {
        size_t n = 0;
        cb_fir_f64_state_len(h_, &n);
        std::vector<c64> s(n);
        cb_fir_f64_get_state(h_, reinterpret_cast<double *>(s.data()), n);
        return s;
    }
};

// BatchFirNode<Complex<f64>>::new(taps, state) / run(&[Complex<f64>])   src/filter/fir_node.rs:193-220
struct BatchFirNodeF64 : Node1<BatchFirNodeF64, std::vector<c64>, std::vector<c64>>, FirF64Handle {
    BatchFirNodeF64(const std::vector<c64> &taps, const std::vector<c64> *state = nullptr, uint32_t decim = 1,
                    uint32_t interp = 1)
        : FirF64Handle(taps, state, decim, interp) {}
    Result<std::vector<c64>> run(const std::vector<c64> &in) { return filter(in.data(), in.size()); }
};

// PulseNode<f64>::new(taps, sam_per_sym) / run(&Complex<f64>) -> Vec   src/pulse.rs:71-92
struct PulseNodeF64 : Node1<PulseNodeF64, c64, std::vector<c64>>, FirF64Handle {
    PulseNodeF64(const std::vector<c64> &taps, size_t sam_per_sym) : FirF64Handle(taps, nullptr, 1, (uint32_t)sam_per_sym) {}
    Result<std::vector<c64>> run(const c64 &sym) { return filter(&sym, 1); }
};

// FFTBatchNode::new(fft_size, ifft) / run(&[Complex<T>])      src/fft/fft_node.rs:65-83
struct FFTBatchNode : Node1<FFTBatchNode, std::vector<c32>, std::vector<c32>> {
    cb_fft *h_ = nullptr;
    FFTBatchNode(size_t fft_size, bool ifft)
    {
        if (cb_fft_create(fft_size, ifft, &h_)) throw std::runtime_error(cb_last_error());
    }
    ~FFTBatchNode() { cb_fft_destroy(h_); }
    Result<std::vector<c32>> run(const std::vector<c32> &in)
    {
        std::vector<c32> out(in.size());
        int st = cb_fft_run(h_, reinterpret_cast<const float *>(in.data()), in.size(), reinterpret_cast<float *>(out.data()));
        return st ? Result<std::vector<c32>>::Err(map_status(st)) : Result<std::vector<c32>>::Ok(std::move(out));
    }
};

// FFTBatchNode<Complex<f64>>: the reference runs every transform in f64 (src/fft/mod.rs:73-96); see cb_fft_f64
struct FFTBatchNodeF64 : Node1<FFTBatchNodeF64, std::vector<c64>, std::vector<c64>> {
    cb_fft_f64 *h_ = nullptr;
    FFTBatchNodeF64(size_t fft_size, bool ifft)
    {
        if (cb_fft_f64_create(fft_size, ifft, &h_)) throw std::runtime_error(cb_last_error());
    }
    ~FFTBatchNodeF64() { cb_fft_f64_destroy(h_); }
    FFTBatchNodeF64(const FFTBatchNodeF64 &) = delete;
    FFTBatchNodeF64 &operator=(const FFTBatchNodeF64 &) = delete;
    Result<std::vector<c64>> run(const std::vector<c64> &in)
    {
        std::vector<c64> out(in.size());
        int st = cb_fft_f64_run(h_, reinterpret_cast<const double *>(in.data()), in.size(),
                                reinterpret_cast<double *>(out.data()));
        return st ? Result<std::vector<c64>>::Err(map_status(st)) : Result<std::vector<c64>>::Ok(std::move(out));
    }
};

// FFTSampleNode (#[aggregate]): emits only when fft_size samples have arrived   src/fft/fft_node.rs:101-168
struct FFTSampleNode : Node1<FFTSampleNode, c32, std::vector<c32>, true> {
    cb_fft *h_ = nullptr;
    size_t fft_size;
    std::vector<c32> samples;
    FFTSampleNode(size_t n, bool ifft) : fft_size(n)
    {
        if (cb_fft_create(n, ifft, &h_)) throw std::runtime_error(cb_last_error());
    }
    ~FFTSampleNode() { cb_fft_destroy(h_); }
    Result<std::optional<std::vector<c32>>> run(const c32 &s)
    {
        using R = Result<std::optional<std::vector<c32>>>;
        samples.push_back(s);
        if (samples.size() < fft_size) return R::Ok(std::nullopt);
        std::vector<c32> out(fft_size);
        int st = cb_fft_run(h_, reinterpret_cast<const float *>(samples.data()), fft_size, reinterpret_cast<float *>(out.data()));
        samples.clear();
        return st ? R::Err(map_status(st)) : R::Ok(std::optional<std::vector<c32>>(std::move(out)));
    }
};

// FMDemodNode::new() / run(&[Complex<T>]) -> Vec<T>           src/modulation/analog_node.rs:43-52
struct FMDemodNode : Node1<FMDemodNode, std::vector<c32>, std::vector<float>> {
    cb_fm *h_ = nullptr;
    FMDemodNode() { if (cb_fm_create(&h_)) throw std::runtime_error(cb_last_error()); }
    ~FMDemodNode() { cb_fm_destroy(h_); }
    Result<std::vector<float>> run(const std::vector<c32> &in)
    {
        std::vector<float> out(in.size());
        int st = cb_fm_run(h_, reinterpret_cast<const float *>(in.data()), in.size(), out.data());
        return st ? Result<std::vector<float>>::Err(map_status(st)) : Result<std::vector<float>>::Ok(std::move(out));
    }
};

// ------------------------------------------------------------------ device-resident edges
// What crosses a channel between two GPU nodes instead of a Vec: a ref-counted handle to a pooled pinned-host or
// device buffer (Clone = cb_buf_retain, Drop = cb_buf_release; the derive macro clones once per downstream edge,
// node_derive/src/lib.rs:156).  `len` = valid elements.  The producer records `ready` on its stream, the consumer
// makes its stream wait for it and records `done` behind its own use before dropping the message, so no node ever
// blocks the host and the pool never hands a block to its next owner early.
class Buf {
    cb_buf *b_ = nullptr;
public:
    size_t len = 0;
    Buf() = default;
    Buf(cb_buf *b, size_t n) : b_(b), len(n) {}
    Buf(const Buf &o) : b_(o.b_), len(o.len) { if (b_) cb_buf_retain(b_); }
    Buf(Buf &&o) noexcept : b_(o.b_), len(o.len) { o.b_ = nullptr; }
    Buf &operator=(const Buf &o) { if (this != &o) { if (b_) cb_buf_release(b_); b_ = o.b_; len = o.len; if (b_) cb_buf_retain(b_); } return *this; }
    Buf &operator=(Buf &&o) noexcept { if (this != &o) { if (b_) cb_buf_release(b_); b_ = o.b_; len = o.len; o.b_ = nullptr; } return *this; }
    ~Buf() { if (b_) cb_buf_release(b_); }
    static Buf device(size_t bytes, size_t n) { cb_buf *b = nullptr; if (cb_buf_alloc_device(bytes, &b)) throw std::runtime_error(cb_last_error()); return Buf(b, n); }
    static Buf pinned(size_t bytes, size_t n) { cb_buf *b = nullptr; if (cb_buf_alloc_pinned(bytes, &b)) throw std::runtime_error(cb_last_error()); return Buf(b, n); }
    void *ptr() const { return cb_buf_ptr(b_); }
    cb_buf *raw() const { return b_; }
};

struct StreamOwner {
    cb_stream *st = nullptr;
    StreamOwner() { if (cb_stream_create(&st)) throw std::runtime_error(cb_last_error()); }
    ~StreamOwner() { cb_stream_destroy(st); }
    void *s() const { return cb_stream_handle(st); }
};

// graph edge host -> device: pinned message in, device message out (elem = bytes per element)
struct H2DNode : Node1<H2DNode, Buf, Buf>, StreamOwner {
    size_t elem;
    explicit H2DNode(size_t elem_bytes) : elem(elem_bytes) {}
    Result<Buf> run(const Buf &in)
    {
        Buf out = Buf::device(in.len * elem, in.len);
        int st = cb_copy_h2d_async(out.ptr(), in.ptr(), in.len * elem, s());
        if (!st) st = cb_buf_record_done(in.raw(), s());
        if (!st) st = cb_buf_record_ready(out.raw(), s());
        return st ? Result<Buf>::Err(map_status(st)) : Result<Buf>::Ok(std::move(out));
    }
};

// graph edge device -> host
struct D2HNode : Node1<D2HNode, Buf, Buf>, StreamOwner {
    size_t elem;
    explicit D2HNode(size_t elem_bytes) : elem(elem_bytes) {}
    Result<Buf> run(const Buf &in)
    {
        Buf out = Buf::pinned(in.len * elem, in.len);
        int st = cb_buf_wait_ready(in.raw(), s());
        if (!st) st = cb_copy_d2h_async(out.ptr(), in.ptr(), in.len * elem, s());
        if (!st) st = cb_buf_record_done(in.raw(), s());
        if (!st) st = cb_buf_record_ready(out.raw(), s());
        return st ? Result<Buf>::Err(map_status(st)) : Result<Buf>::Ok(std::move(out));
    }
};

// BatchFirNode between device edges (complex f32 in and out; decim / interp fused)
struct BatchFirDevNode : Node1<BatchFirDevNode, Buf, Buf>, FirHandle {
    BatchFirDevNode(const std::vector<c32> &taps, const std::vector<c32> *state = nullptr, uint32_t decim = 1, uint32_t interp = 1)
        : FirHandle(taps, state, decim, interp) {}
    Result<Buf> run(const Buf &in)
    {
        size_t no = 0;
        cb_fir_out_len(h_, in.len, &no);
        Buf out = Buf::device(no * sizeof(c32), no);
        void *s = cb_fir_stream(h_);
        int st = cb_buf_wait_ready(in.raw(), s);
        if (!st) st = cb_fir_run_dev(h_, static_cast<const float *>(in.ptr()), in.len, static_cast<float *>(out.ptr()), no, &no, s);
        if (!st) st = cb_buf_record_done(in.raw(), s);
        if (!st) st = cb_buf_record_ready(out.raw(), s);
        return st ? Result<Buf>::Err(map_status(st)) : Result<Buf>::Ok(std::move(out));
    }
};

// Convert2Node -> BatchFirNode -> Convert3Node -> DecimateNode of examples/fm_radio.rs:98-164 between device edges
struct FirRealDevNode : Node1<FirRealDevNode, Buf, Buf>, FirHandle {
    FirRealDevNode(const std::vector<c32> &taps, uint32_t decim) : FirHandle(taps, nullptr, decim, 1) {}
    Result<Buf> run(const Buf &in)
    {
        size_t no = 0;
        cb_fir_out_len(h_, in.len, &no);
        Buf out = Buf::device(no * sizeof(float), no);
        void *s = cb_fir_stream(h_);
        int st = cb_buf_wait_ready(in.raw(), s);
        if (!st) st = cb_fir_run_real_dev(h_, static_cast<const float *>(in.ptr()), in.len, static_cast<float *>(out.ptr()), no, &no, s);
        if (!st) st = cb_buf_record_done(in.raw(), s);
        if (!st) st = cb_buf_record_ready(out.raw(), s);
        return st ? Result<Buf>::Err(map_status(st)) : Result<Buf>::Ok(std::move(out));
    }
};

// ConvertNode -> filt1 -> dec1 -> FMDemodNode of examples/fm_radio.rs:84-97,144-160 on raw u8 IQ, one channel
struct FmFrontDevNode : Node1<FmFrontDevNode, Buf, Buf>, StreamOwner {
    cb_chain *h_ = nullptr;
    FmFrontDevNode(const std::vector<c32> &taps, uint32_t decim)
    {
        if (cb_chain_create(1, nullptr, nullptr, reinterpret_cast<const float *>(taps.data()), taps.size(), decim, 1, &h_))
            throw std::runtime_error(cb_last_error());
    }
    ~FmFrontDevNode() { cb_chain_destroy(h_); }
    Result<Buf> run(const Buf &in)  // in.len = IQ byte pairs
    {
        size_t no = 0;
        cb_chain_out_len(h_, in.len, &no);
        Buf out = Buf::device(no * sizeof(float), no);
        int st = cb_buf_wait_ready(in.raw(), s());
        if (!st) st = cb_chain_run_u8_dev(h_, static_cast<const uint8_t *>(in.ptr()), in.len, static_cast<float *>(out.ptr()), no, &no, s());
        if (!st) st = cb_buf_record_done(in.raw(), s());
        if (!st) st = cb_buf_record_ready(out.raw(), s());
        return st ? Result<Buf>::Err(map_status(st)) : Result<Buf>::Ok(std::move(out));
    }
};

// rrc_taps::<f32> (src/util/math.rs:221-280); empty Result.err == InvalidRolloffError for beta outside [0, 1]
inline bool rrc_taps(uint32_t n_taps, double sam_per_sym, double beta, std::vector<c32> &taps)
{
    taps.assign(n_taps, c32(0.f, 0.f));
    return cb_rrc_taps(n_taps, sam_per_sym, beta, reinterpret_cast<float *>(taps.data())) == CB_OK;
}

// TimingEstimatorNode (src/demodulation/timing_estimator.rs:116-137): Vec<Complex<f64>> in, f64 out
struct TimingEstimatorNode : Node1<TimingEstimatorNode, std::vector<std::complex<double>>, double> {
    cb_timing *h = nullptr;
    bool ok = false;  // false: MathError::InvalidRolloffError (or no device)
    TimingEstimatorNode(uint32_t n, uint32_t d, double alpha) { ok = cb_timing_create(n, d, alpha, &h) == CB_OK; }
    ~TimingEstimatorNode() { cb_timing_destroy(h); }
    TimingEstimatorNode(const TimingEstimatorNode &) = delete;
    TimingEstimatorNode &operator=(const TimingEstimatorNode &) = delete;
    Result<double> run(const std::vector<std::complex<double>> &in)
    {
        double est = 0.0;
        int st = cb_timing_push(h, reinterpret_cast<const double *>(in.data()), in.size(), &est);
        return st ? Result<double>::Err(map_status(st)) : Result<double>::Ok(est);
    }
};

// frequency_offset_estimate (src/demodulation/frequency_estimator.rs:27-42)
inline Result<double> frequency_offset_estimate(const std::vector<std::complex<double>> &samples)
{
    double est = 0.0;
    int st = cb_freq_estimate(reinterpret_cast<const double *>(samples.data()), samples.size(), &est);
    return st ? Result<double>::Err(map_status(st)) : Result<double>::Ok(est);
}

}  // namespace comms_b200
