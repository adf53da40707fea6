// C ABI of libcomms_b200.so (see include/comms_b200.h): handles, buffers, streams,
// host-pointer pipelines.  No torch, no C++ types in any signature, no CPU fallback.
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <map>
#include <mutex>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>
#include <vector>

#include "chain_kernels.cuh"
#include "common.cuh"
#include "estimator_kernels.cuh"
#include "fft_kernels.cuh"
#include "fft64_core.cuh"
#include "fft_f64_kernels.cuh"
#include "fir_f64_kernels.cuh"
#include "fir_kernels.cuh"
#include "misc_kernels.cuh"

namespace cb {

static thread_local char g_err[512] = "";
static thread_local int g_dev = 0;

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return CB_ERR_NO_DEVICE;
    if (e == cudaErrorMemoryAllocation) return CB_ERR_OOM;
    return CB_ERR_CUDA;
}

int current_device() { return g_dev; }

static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

static int use_device(int dev)
{
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        (void)cudaGetLastError();
        set_error("no CUDA device available (%s); libcomms_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return CB_ERR_NO_DEVICE;
    }
    CB_REQUIRE(dev >= 0 && dev < count, CB_ERR_INVALID_ARG, "device %d out of range (0..%d)", dev, count - 1);
    CB_CUDA(cudaSetDevice(dev));
    return CB_OK;
}

int ensure_device() { return use_device(g_dev); }

// Parallel host memcpy for the pageable-memory path of the host-pointer entries.  A Rust `Vec` (what the reference's
// run(&[Complex<T>]) -> Vec<Complex<T>> hands over) is pageable: cudaMemcpyAsync from it goes through the driver's own
// single-threaded staging copy and serialises with the kernels (measured: 0.8 instead of 5.9 Gsamples/s for a 2 GiB
// call).  Large pageable calls are staged by this pool instead: each chunk is copied into / out of a pinned slot of the
// handle's lane by COMMS_B200_STAGE_THREADS threads (default min(8, cores/2)) while the previous chunk's DMA and kernel run.
class StagePool {
    struct Task {
        char *dst;
        const char *src;
        size_t bytes;
    };
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv, done_cv;
    std::vector<Task> q;
    size_t pending = 0;
    bool stop = false;

    void worker()
    {
        for (;;) {
            Task t;
            {
                std::unique_lock<std::mutex> l(m);
                cv.wait(l, [&] { return stop || !q.empty(); });
                if (q.empty()) return;
                t = q.back();
                q.pop_back();
            }
            memcpy(t.dst, t.src, t.bytes);
            {
                std::lock_guard<std::mutex> l(m);
                --pending;
            }
            done_cv.notify_all();
        }
    }

public:
    StagePool()
    {
        unsigned n = std::thread::hardware_concurrency() / 2;
        if (n > 8) n = 8;
        if (const char *e = getenv("COMMS_B200_STAGE_THREADS")) n = (unsigned)atoi(e);
        if (n < 1) n = 1;
        if (n > 64) n = 64;
        for (unsigned i = 1; i < n; ++i) th.emplace_back([this] { worker(); });  // the caller is the n-th copier
    }
    ~StagePool()
    {
        {
            std::lock_guard<std::mutex> l(m);
            stop = true;
        }
        cv.notify_all();
        for (auto &t : th) t.join();
    }
    // blocking copy; safe to call from several node threads at once (they share the workers)
    void copy(void *dst, const void *src, size_t bytes)
    {
        const size_t parts = th.size() + 1;
        const size_t piece = round_up(ceil_div(bytes, parts), (size_t)4096);
        if (th.empty() || bytes < ((size_t)1 << 20)) {
            memcpy(dst, src, bytes);
            return;
        }
        size_t mine_off = 0, mine_len = piece < bytes ? piece : bytes, posted = 0;
        {
            std::lock_guard<std::mutex> l(m);
            for (size_t off = mine_len; off < bytes; off += piece) {
                q.push_back(Task{(char *)dst + off, (const char *)src + off, bytes - off < piece ? bytes - off : piece});
                ++posted;
            }
            pending += posted;
        }
        cv.notify_all();
        memcpy((char *)dst + mine_off, (const char *)src + mine_off, mine_len);
        std::unique_lock<std::mutex> l(m);
        // `pending` counts every caller's pieces; waiting for zero is conservative but always correct
        done_cv.wait(l, [&] { return pending == 0; });
    }
};

static StagePool &stage_pool()
{
    static StagePool p;
    return p;
}

// pageable (unregistered) host memory?  Pinned / registered / managed memory takes the direct DMA path.
static bool is_pageable(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

// Pageable calls of at least this many bytes are staged through the handle's pinned slots.  Default 0: also the small
// messages the reference's graphs pass around (a 4096-symbol BPSK message is 32 KiB in, 128 KiB out) -- the driver's own
// path for a pageable copy blocks in the D2H call and costs 82 us per such message, a memcpy into / out of a pinned slot
// around two asynchronous DMAs and one wait costs less than half (profiles/r03p_bench_graph.jsonl).  Pieces below 1 MiB
// are copied by the calling thread, larger ones by the pool.  COMMS_B200_STAGE_MIN_BYTES overrides.
// device-side address of pinned / registered / managed host memory, or NULL (pageable, or not mapped)
template <typename T>
static const T *host_device_view(const T *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    if (a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged) return static_cast<const T *>(a.devicePointer);
    return nullptr;
}

// host-pointer FIR calls whose input + output fit in this many bytes run as one kernel over pinned host memory
static const size_t ZEROCOPY_MAX_BYTES = [] {
    const char *e = getenv("COMMS_B200_ZEROCOPY_MAX_BYTES");
    return e ? (size_t)atoll(e) : (size_t)1 << 20;
}();

static const size_t STAGE_MIN_BYTES = [] {
    const char *e = getenv("COMMS_B200_STAGE_MIN_BYTES");
    return e ? (size_t)atoll(e) : (size_t)0;
}();

// Two copy/compute lanes used by the host-pointer entry points: chunk i runs
// H2D -> kernel -> D2H on lane i%2, so the copy engines and the SMs overlap.
struct HostPipe {
    cudaStream_t lane[2] = {nullptr, nullptr};
    void *in[2] = {nullptr, nullptr};
    void *out[2] = {nullptr, nullptr};
    size_t in_cap = 0, out_cap = 0;
    void *aux_in[2] = {nullptr, nullptr}, *aux_out[2] = {nullptr, nullptr};  // f32 sides of the i16-IQ entries
    size_t aux_in_cap = 0, aux_out_cap = 0;
    // pinned staging slots for pageable callers (allocated on first use), one per lane and direction
    void *pin_in[2] = {nullptr, nullptr}, *pin_out[2] = {nullptr, nullptr};
    size_t pin_in_cap = 0, pin_out_cap = 0;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    bool in_busy[2] = {false, false};
    void *pend_dst[2] = {nullptr, nullptr};
    size_t pend_bytes[2] = {0, 0};
    bool stage_in = false, stage_out = false;

    int init(cudaStream_t first)
    {
        lane[0] = first;
        CB_CUDA(cudaStreamCreateWithFlags(&lane[1], cudaStreamNonBlocking));
        return CB_OK;
    }
    int reserve(size_t in_bytes, size_t out_bytes)
    {
        if (in_bytes > in_cap) {
            for (int i = 0; i < 2; ++i) {
                if (in[i]) CB_CUDA(cudaFree(in[i]));
                in[i] = nullptr;
                CB_CUDA(cudaMalloc(&in[i], in_bytes));
            }
            in_cap = in_bytes;
        }
        if (out_bytes > out_cap) {
            for (int i = 0; i < 2; ++i) {
                if (out[i]) CB_CUDA(cudaFree(out[i]));
                out[i] = nullptr;
                CB_CUDA(cudaMalloc(&out[i], out_bytes));
            }
            out_cap = out_bytes;
        }
        return CB_OK;
    }
    int reserve_aux(size_t in_bytes, size_t out_bytes)
    {
        if (in_bytes > aux_in_cap) {
            for (int i = 0; i < 2; ++i) {
                if (aux_in[i]) CB_CUDA(cudaFree(aux_in[i]));
                aux_in[i] = nullptr;
                CB_CUDA(cudaMalloc(&aux_in[i], in_bytes));
            }
            aux_in_cap = in_bytes;
        }
        if (out_bytes > aux_out_cap) {
            for (int i = 0; i < 2; ++i) {
                if (aux_out[i]) CB_CUDA(cudaFree(aux_out[i]));
                aux_out[i] = nullptr;
                CB_CUDA(cudaMalloc(&aux_out[i], out_bytes));
            }
            aux_out_cap = out_bytes;
        }
        return CB_OK;
    }
    // Decide per call whether the caller's buffers are staged (large and pageable) and size the pinned slots.
    int begin_call(const void *host_in, size_t total_in, size_t chunk_in, void *host_out, size_t total_out, size_t chunk_out)
    {
        stage_in = total_in >= STAGE_MIN_BYTES && is_pageable(host_in);
        stage_out = total_out >= STAGE_MIN_BYTES && is_pageable(host_out);
        for (int i = 0; i < 2; ++i) {
            in_busy[i] = false;
            pend_dst[i] = nullptr;
        }
        if (stage_in && chunk_in > pin_in_cap) {
            for (int i = 0; i < 2; ++i) {
                if (pin_in[i]) CB_CUDA(cudaFreeHost(pin_in[i]));
                pin_in[i] = nullptr;
                CB_CUDA(cudaMallocHost(&pin_in[i], chunk_in));
            }
            pin_in_cap = chunk_in;
        }
        if (stage_out && chunk_out > pin_out_cap) {
            for (int i = 0; i < 2; ++i) {
                if (pin_out[i]) CB_CUDA(cudaFreeHost(pin_out[i]));
                pin_out[i] = nullptr;
                CB_CUDA(cudaMallocHost(&pin_out[i], chunk_out));
            }
            pin_out_cap = chunk_out;
        }
        for (int i = 0; i < 2; ++i) {
            if ((stage_in || stage_out) && !ev_in[i]) CB_CUDA(cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming));
            if ((stage_in || stage_out) && !ev_out[i]) CB_CUDA(cudaEventCreateWithFlags(&ev_out[i], cudaEventDisableTiming));
        }
        return CB_OK;
    }
    int h2d(int l, void *dev_dst, const void *host_src, size_t bytes)
    {
        if (!stage_in) {
            CB_CUDA(cudaMemcpyAsync(dev_dst, host_src, bytes, cudaMemcpyHostToDevice, lane[l]));
            return CB_OK;
        }
        if (in_busy[l]) CB_CUDA(cudaEventSynchronize(ev_in[l]));  // the slot's previous DMA has left it
        stage_pool().copy(pin_in[l], host_src, bytes);
        CB_CUDA(cudaMemcpyAsync(dev_dst, pin_in[l], bytes, cudaMemcpyHostToDevice, lane[l]));
        CB_CUDA(cudaEventRecord(ev_in[l], lane[l]));
        in_busy[l] = true;
        return CB_OK;
    }
    int flush_out(int l)
    {
        if (!pend_dst[l]) return CB_OK;
        CB_CUDA(cudaEventSynchronize(ev_out[l]));
        stage_pool().copy(pend_dst[l], pin_out[l], pend_bytes[l]);
        pend_dst[l] = nullptr;
        return CB_OK;
    }
    int d2h(int l, void *host_dst, const void *dev_src, size_t bytes)
    {
        if (!stage_out) {
            CB_CUDA(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, lane[l]));
            return CB_OK;
        }
        int rc = flush_out(l);
        if (rc) return rc;
        CB_CUDA(cudaMemcpyAsync(pin_out[l], dev_src, bytes, cudaMemcpyDeviceToHost, lane[l]));
        CB_CUDA(cudaEventRecord(ev_out[l], lane[l]));
        pend_dst[l] = host_dst;
        pend_bytes[l] = bytes;
        return CB_OK;
    }
    int sync()
    {
        // drain the staged outputs in issue order (the older lane first) while the other lane's DMA still runs
        if (stage_out) {
            for (int i = 0; i < 2; ++i) {
                int rc = flush_out(i);
                if (rc) return rc;
            }
        }
        CB_CUDA(cudaStreamSynchronize(lane[0]));
        CB_CUDA(cudaStreamSynchronize(lane[1]));
        return CB_OK;
    }
    void destroy()
    {
        for (int i = 0; i < 2; ++i) {
            if (in[i]) cudaFree(in[i]);
            if (out[i]) cudaFree(out[i]);
            if (aux_in[i]) cudaFree(aux_in[i]);
            if (aux_out[i]) cudaFree(aux_out[i]);
            if (pin_in[i]) cudaFreeHost(pin_in[i]);
            if (pin_out[i]) cudaFreeHost(pin_out[i]);
            if (ev_in[i]) cudaEventDestroy(ev_in[i]);
            if (ev_out[i]) cudaEventDestroy(ev_out[i]);
        }
        if (lane[1]) cudaStreamDestroy(lane[1]);
    }
};

// Per-handle ordering of carried state across streams.  *_run_dev may be given any stream, while the handle's carried
// state (history / phase / prev double buffers, the FFT scratch ring and its counters) is one set of device buffers:
// every launch records `ev` behind itself, and the next use on ANOTHER stream (or a host-side get/set/destroy) waits
// for it, so two calls on different streams are ordered exactly like two calls on one stream.
struct LastUse {
    cudaEvent_t ev = nullptr;
    cudaStream_t s = nullptr;
    bool has = false;
    int begin(cudaStream_t cur)
    {
        if (has && cur != s) CB_CUDA(cudaStreamWaitEvent(cur, ev, 0));
        return CB_OK;
    }
    int end(cudaStream_t cur)
    {
        if (!ev) CB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CB_CUDA(cudaEventRecord(ev, cur));
        s = cur;
        has = true;
        return CB_OK;
    }
    int sync()
    {
        if (has) CB_CUDA(cudaEventSynchronize(ev));
        return CB_OK;
    }
    void destroy()
    {
        if (ev) {
            if (has) cudaEventSynchronize(ev);
            cudaEventDestroy(ev);
            ev = nullptr;
        }
    }
};

// [a, a+na) and [b, b+nb) share a byte.  The filter / chain / FM kernels read halo samples that other CTAs own and
// rebuild the carried history from the input after other CTAs may have stored their outputs, so an in-place (or
// overlapping) call would silently corrupt both the samples and the state of every later batch.
static inline bool ranges_overlap(const void *a, size_t na, const void *b, size_t nb)
{
    const uintptr_t a0 = (uintptr_t)a, b0 = (uintptr_t)b;
    return a0 < b0 + nb && b0 < a0 + na;
}
#define CB_NO_ALIAS(in, in_bytes, out, out_bytes, who)                                                       \
    CB_REQUIRE(!ranges_overlap((in), (in_bytes), (out), (out_bytes)), CB_ERR_INVALID_ARG,                    \
               who ": input and output ranges overlap (in-place calls are not provided: the kernel reads "   \
                   "neighbouring tiles' samples and rebuilds the carried state from the input)")

// complex samples per pipelined chunk of the host-pointer entries (default 2^22 = 32 MiB; COMMS_B200_HOST_CHUNK_LOG2)
static const size_t HOST_CHUNK = [] {
    const char *e = getenv("COMMS_B200_HOST_CHUNK_LOG2");
    const int l = e ? atoi(e) : 22;
    return (size_t)1 << (l >= 12 && l <= 30 ? l : 22);
}();

// ---------------------------------------------------------------------------------------------------- buffer pool
// cb_buf_alloc_* used to be one cudaMalloc / cudaMallocHost per message and one cudaFree per release: a device
// synchronisation per message.  Blocks now come from a size-classed, thread-safe free list per (device, kind), and the
// pool applies BACK-PRESSURE: the reference's channels are unbounded (src/node/mod.rs:152), so a source that runs
// ahead of a GPU node would otherwise queue pinned / device buffers without limit.  While the bytes handed out and
// not yet released exceed the high-water mark, cb_pool_throttle() -- called by the nodes where pool buffers start --
// blocks until releases bring them back under it (or fails with CB_ERR_OOM after the timeout, so that a graph that
// can never release does not hang forever).
struct BufPool {
    struct Block {
        void *ptr;
        std::vector<cudaEvent_t> pending;  // uses recorded by the previous owner; waited for when the block is reused
        cudaEvent_t spare_ready;           // the previous owner's event objects, recycled with the block
        std::vector<cudaEvent_t> spare_done;
    };
    std::mutex m;
    std::condition_variable cv;
    std::map<size_t, std::vector<Block>> free_list;  // size class -> blocks
    size_t live = 0, cached = 0;
    size_t max_live = 0;      // 0 = unlimited
    size_t max_cached = (size_t)1 << 30;
    int timeout_ms = 10000;
    uint64_t hits = 0, misses = 0, waits = 0;
};
static BufPool g_pools[16][2];  // [device][is_device]

static size_t pool_class(size_t bytes)
{
    if (bytes <= 256) return 256;
    if (bytes <= ((size_t)1 << 20)) {
        size_t c = 256;
        while (c < bytes) c <<= 1;
        return c;
    }
    return round_up(bytes, (size_t)2 << 20);
}

static BufPool &pool_of(int device, int is_device) { return g_pools[device & 15][is_device ? 1 : 0]; }

}  // namespace cb

using namespace cb;

// ============================================================================ handles
struct cb_stream {
    int device;
    cudaStream_t s;
};

struct cb_buf {
    std::atomic<int> refs;
    void *ptr;
    size_t bytes;      // as requested
    size_t cls_bytes;  // size class actually allocated (what the pool accounts)
    int is_device;
    int device;
    cudaEvent_t ready;  // recorded by the producing node's stream (cb_buf_record_ready)
    bool has_ready;
    std::vector<cudaEvent_t> done;  // recorded by consumers behind their last use (cb_buf_record_done)
    size_t n_done;                  // how many of `done` are recorded for the current owner
};

struct cb_fir {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    std::vector<float2> taps;  // as given
    float2 *taps_dev;
    size_t nstate;     // reference state length (zero-stuffed domain when interp > 1)
    uint32_t k_eff;    // min(ntaps, nstate)
    bool taps_real;
    uint32_t decim, interp;
    uint32_t hist_len;  // input-domain samples kept
    float2 *hist[2];
    int cur;
    void *tc_img;       // tensor-core path: prepacked tap image (device), or NULL
    FirTcPlan tc;
    FirFix fix[2];      // exact fall-back work lists of the tensor-core path, one per host-pipeline lane
    float2 *qscratch;   // f32 result of the unfused cb_fir_run_dev_i16 path, grown on demand
    size_t qscratch_len;
    float2 *rscratch;   // unfused cb_fir_run_real_dev path: widened input followed by the complex result
    size_t rscratch_len;
    // overlap-save path for 129 .. 1025 taps: taps' spectrum, the two 4096-point twiddle tables, frame spectra
    float2 *ols_hf, *ols_twf, *ols_twi, *ols_spec;
    size_t ols_spec_frames;
    LastUse last;
};

struct cb_mixer {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    double phase, dphase;
};

struct cb_fft {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    FftPlanDev plan;
    float2 *tw, *tw1, *tw2, *tw16, *tw16a, *tw16b, *scratch;
    // FFT_BLUESTEIN (any other size): chirp w[n] (n entries), transform of the wrapped conj chirp (bl_m entries),
    // forward / inverse power-of-two plans of bl_m points, two work buffers of bl_frames frames of bl_m points
    cb_fft *sub_f, *sub_i;
    float2 *chirp, *bspec, *bufa, *bufb;
    size_t bl_m, bl_frames;
    LastUse last;
};

struct cb_fm {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    float2 *prev[2];
    int cur;
    LastUse last;
};

struct cb_chain {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    size_t channels;
    bool mix, fm, cplx;
    ChainTaps taps;
    uint32_t ntaps, decim, hist_len;
    double *phase[2], *dphase;
    float2 *hist[2], *prev[2];
    int cur;
    float2 *cscratch;   // converted input of the unfused cb_chain_run_u8 path, grown on demand
    size_t cscratch_len;
    void *tc_img;       // tensor-core byte front end: prepacked tap image (device), or NULL
    float tc_inv_scale, tc_dc;
    float2 *tc_seam;    // its per-tile first / last outputs, grown on demand
    size_t tc_seam_len;
    LastUse last;
};

static inline cudaStream_t pick_stream(void *user, cudaStream_t own) { return user ? (cudaStream_t)user : own; }

extern "C" {

// ============================================================================ library
int cb_version(void) { return 1000 * 0 + 1; }
const char *cb_last_error(void) { return g_err; }

const char *cb_status_str(int st)
{
    switch (st) {
    case CB_OK: return "ok";
    case CB_ERR_INVALID_ARG: return "invalid argument";
    case CB_ERR_SIZE: return "size mismatch";
    case CB_ERR_CUDA: return "CUDA failure";
    case CB_ERR_NO_DEVICE: return "no CUDA device";
    case CB_ERR_OOM: return "out of memory";
    case CB_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown status";
    }
}

int cb_device_count(int *count)
{
    CB_REQUIRE(count, CB_ERR_INVALID_ARG, "count is NULL");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        c = 0;
    }
    *count = c;
    return CB_OK;
}

int cb_launch_count(uint64_t *count)
{
    CB_REQUIRE(count, CB_ERR_INVALID_ARG, "count is NULL");
    *count = g_launches.load(std::memory_order_relaxed);
    return CB_OK;
}

int cb_init(int device)
{
    int rc = use_device(device);
    if (rc) return rc;
    g_dev = device;
    CB_CUDA(cudaFree(nullptr));  // force context creation
    return CB_OK;
}

int cb_device_synchronize(void)
{
    int rc = ensure_device();
    if (rc) return rc;
    CB_CUDA(cudaDeviceSynchronize());
    return CB_OK;
}

// ============================================================================ streams
int cb_stream_create(cb_stream **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    int rc = ensure_device();
    if (rc) return rc;
    cb_stream *s = new (std::nothrow) cb_stream;
    CB_REQUIRE(s, CB_ERR_OOM, "host allocation failed");
    s->device = g_dev;
    cudaError_t e = cudaStreamCreateWithFlags(&s->s, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete s;
        return cuda_fail(e, "cudaStreamCreateWithFlags", __FILE__, __LINE__);
    }
    *out = s;
    return CB_OK;
}

int cb_stream_destroy(cb_stream *s)
{
    if (!s) return CB_OK;
    cudaSetDevice(s->device);
    cudaStreamDestroy(s->s);
    delete s;
    return CB_OK;
}

int cb_stream_sync(cb_stream *s)
{
    CB_REQUIRE(s, CB_ERR_INVALID_ARG, "stream is NULL");
    CB_CUDA(cudaSetDevice(s->device));
    CB_CUDA(cudaStreamSynchronize(s->s));
    return CB_OK;
}

void *cb_stream_handle(cb_stream *s) { return s ? (void *)s->s : nullptr; }

// ============================================================================ buffers
static int buf_alloc(size_t bytes, int is_device, cb_buf **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    int rc = ensure_device();
    if (rc) return rc;
    cb_buf *b = new (std::nothrow) cb_buf;
    CB_REQUIRE(b, CB_ERR_OOM, "host allocation failed");
    b->refs.store(1);
    b->bytes = bytes;
    b->cls_bytes = pool_class(bytes);
    b->is_device = is_device;
    b->device = g_dev;
    b->ptr = nullptr;
    b->ready = nullptr;
    b->has_ready = false;
    b->n_done = 0;
    BufPool &p = pool_of(g_dev, is_device);
    BufPool::Block blk{nullptr, {}, nullptr, {}};
    bool have = false;
    {
        std::unique_lock<std::mutex> l(p.m);
        auto it = p.free_list.find(b->cls_bytes);
        if (it != p.free_list.end() && !it->second.empty()) {
            blk = std::move(it->second.back());
            it->second.pop_back();
            p.cached -= b->cls_bytes;
            ++p.hits;
            have = true;
        } else {
            ++p.misses;
        }
        p.live += b->cls_bytes;
    }
    if (have) {
        // the previous owner's asynchronous uses must be over before the new owner touches the block
        for (cudaEvent_t e : blk.pending) cudaEventSynchronize(e);
        b->ptr = blk.ptr;
        b->ready = blk.spare_ready;
        b->done = std::move(blk.spare_done);
    } else {
        cudaError_t e = is_device ? cudaMalloc(&b->ptr, b->cls_bytes) : cudaMallocHost(&b->ptr, b->cls_bytes);
        if (e != cudaSuccess) {  // give cached blocks of other classes back to the driver and retry once
            (void)cudaGetLastError();
            cb_pool_trim();
            e = is_device ? cudaMalloc(&b->ptr, b->cls_bytes) : cudaMallocHost(&b->ptr, b->cls_bytes);
        }
        if (e != cudaSuccess) {
            {
                std::lock_guard<std::mutex> l(p.m);
                p.live -= b->cls_bytes;
            }
            p.cv.notify_all();
            delete b;
            return cuda_fail(e, is_device ? "cudaMalloc" : "cudaMallocHost", __FILE__, __LINE__);
        }
    }
    *out = b;
    return CB_OK;
}

int cb_buf_alloc_pinned(size_t bytes, cb_buf **out) { return buf_alloc(bytes, 0, out); }
int cb_buf_alloc_device(size_t bytes, cb_buf **out) { return buf_alloc(bytes, 1, out); }

int cb_buf_retain(cb_buf *b)
{
    CB_REQUIRE(b, CB_ERR_INVALID_ARG, "buffer is NULL");
    b->refs.fetch_add(1);
    return CB_OK;
}

static void block_destroy(BufPool::Block &blk, int is_device)
{
    for (cudaEvent_t e : blk.pending) cudaEventSynchronize(e);
    if (blk.spare_ready) cudaEventDestroy(blk.spare_ready);
    for (cudaEvent_t e : blk.spare_done) cudaEventDestroy(e);
    if (is_device) cudaFree(blk.ptr);
    else cudaFreeHost(blk.ptr);
}

int cb_buf_release(cb_buf *b)
{
    if (!b) return CB_OK;
    if (b->refs.fetch_sub(1) == 1) {
        cudaSetDevice(b->device);
        BufPool &p = pool_of(b->device, b->is_device);
        BufPool::Block blk{b->ptr, {}, b->ready, std::move(b->done)};
        if (b->ready && b->has_ready) blk.pending.push_back(b->ready);  // never reuse (or free) under a pending writer ...
        for (size_t i = 0; i < b->n_done; ++i) blk.pending.push_back(blk.spare_done[i]);  // ... or a pending reader
        bool keep;
        {
            std::lock_guard<std::mutex> l(p.m);
            p.live -= b->cls_bytes;
            keep = p.cached + b->cls_bytes <= p.max_cached;
            if (keep) {
                p.free_list[b->cls_bytes].push_back(std::move(blk));
                p.cached += b->cls_bytes;
            }
        }
        p.cv.notify_all();
        if (!keep) block_destroy(blk, b->is_device);
        delete b;
    }
    return CB_OK;
}

int cb_pool_configure(int is_device, size_t max_live_bytes, size_t max_cached_bytes, int timeout_ms)
{
    int rc = ensure_device();
    if (rc) return rc;
    BufPool &p = pool_of(g_dev, is_device);
    {
        std::lock_guard<std::mutex> l(p.m);
        p.max_live = max_live_bytes;
        p.max_cached = max_cached_bytes;
        if (timeout_ms > 0) p.timeout_ms = timeout_ms;
    }
    p.cv.notify_all();
    return CB_OK;
}

// The back-pressure gate.  Allocations themselves never block (a node in the middle of a graph that waited for a
// buffer while holding one could close a cycle of waits); the nodes where pool buffers START -- a source that fills
// pinned messages, a host->device edge node -- call this once per message before they allocate, holding nothing.
int cb_pool_throttle(int timeout_ms)
{
    for (int kind = 0; kind < 2; ++kind) {
        BufPool &p = pool_of(g_dev, kind);
        std::unique_lock<std::mutex> l(p.m);
        if (!p.max_live || p.live <= p.max_live) continue;
        ++p.waits;
        const int ms = timeout_ms > 0 ? timeout_ms : p.timeout_ms;
        const bool ok = p.cv.wait_for(l, std::chrono::milliseconds(ms), [&] { return !p.max_live || p.live <= p.max_live; });
        if (!ok) {
            const size_t live = p.live, lim = p.max_live;
            l.unlock();
            set_error("buffer pool: %zu bytes of %s messages still in flight against a high-water mark of %zu after %d ms (no "
                      "consumer released a buffer)", live, kind ? "device" : "pinned", lim, ms);
            return CB_ERR_OOM;
        }
    }
    return CB_OK;
}

int cb_pool_stats(int is_device, size_t *live_bytes, size_t *cached_bytes, uint64_t *hits, uint64_t *misses, uint64_t *waits)
{
    BufPool &p = pool_of(g_dev, is_device);
    std::lock_guard<std::mutex> l(p.m);
    if (live_bytes) *live_bytes = p.live;
    if (cached_bytes) *cached_bytes = p.cached;
    if (hits) *hits = p.hits;
    if (misses) *misses = p.misses;
    if (waits) *waits = p.waits;
    return CB_OK;
}

int cb_pool_trim(void)
{
    for (int kind = 0; kind < 2; ++kind) {
        BufPool &p = pool_of(g_dev, kind);
        std::map<size_t, std::vector<BufPool::Block>> take;
        {
            std::lock_guard<std::mutex> l(p.m);
            take.swap(p.free_list);
            p.cached = 0;
        }
        cudaSetDevice(g_dev);
        for (auto &kv : take)
            for (auto &blk : kv.second) block_destroy(blk, kind);
    }
    return CB_OK;
}

void *cb_buf_ptr(cb_buf *b) { return b ? b->ptr : nullptr; }
size_t cb_buf_bytes(cb_buf *b) { return b ? b->bytes : 0; }
int cb_buf_is_device(cb_buf *b) { return b ? b->is_device : 0; }

int cb_buf_record_ready(cb_buf *b, void *stream)
{
    CB_REQUIRE(b, CB_ERR_INVALID_ARG, "buffer is NULL");
    CB_CUDA(cudaSetDevice(b->device));
    if (!b->ready) CB_CUDA(cudaEventCreateWithFlags(&b->ready, cudaEventDisableTiming));
    CB_CUDA(cudaEventRecord(b->ready, (cudaStream_t)stream));
    b->has_ready = true;
    return CB_OK;
}

// A consumer that launched asynchronous work reading (or writing) the buffer records "done" behind it before it drops
// its reference; the pool waits for every such event before the block goes to its next owner.
int cb_buf_record_done(cb_buf *b, void *stream)
{
    CB_REQUIRE(b, CB_ERR_INVALID_ARG, "buffer is NULL");
    CB_CUDA(cudaSetDevice(b->device));
    static std::mutex m;  // several consumers (one per downstream edge) may share the buffer
    std::lock_guard<std::mutex> l(m);
    if (b->n_done == b->done.size()) {
        cudaEvent_t e;
        CB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        b->done.push_back(e);
    }
    CB_CUDA(cudaEventRecord(b->done[b->n_done], (cudaStream_t)stream));
    ++b->n_done;
    return CB_OK;
}

int cb_buf_wait_ready(cb_buf *b, void *stream)
{
    CB_REQUIRE(b, CB_ERR_INVALID_ARG, "buffer is NULL");
    if (!b->has_ready) return CB_OK;
    CB_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, b->ready, 0));
    return CB_OK;
}

int cb_buf_sync(cb_buf *b)
{
    CB_REQUIRE(b, CB_ERR_INVALID_ARG, "buffer is NULL");
    if (!b->has_ready) return CB_OK;
    CB_CUDA(cudaEventSynchronize(b->ready));
    return CB_OK;
}

int cb_copy_h2d_async(void *dst, const void *src, size_t bytes, void *stream)
{
    CB_REQUIRE(dst && src, CB_ERR_INVALID_ARG, "NULL pointer");
    int rc = ensure_device();
    if (rc) return rc;
    CB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return CB_OK;
}

int cb_copy_d2h_async(void *dst, const void *src, size_t bytes, void *stream)
{
    CB_REQUIRE(dst && src, CB_ERR_INVALID_ARG, "NULL pointer");
    int rc = ensure_device();
    if (rc) return rc;
    CB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return CB_OK;
}

// ============================================================================ FIR
// The helpers below serve both FIR handles (cb_fir over float2 samples, cb_fir_f64 over double2): they depend on the
// handle's shape (interp, decim, hist_len) only.
extern "C++" {
template <typename Fir>
static size_t fir_out_len(const Fir *h, size_t n)
{
    const size_t up = n * h->interp;
    return h->decim > 1 ? ceil_div(up, (size_t)h->decim) : up;
}

// reference state (newest first, zero-stuffed domain) -> chronological input-domain history
template <typename Fir, typename T>
static int fir_state_to_hist(const Fir *h, const T *state, size_t nstate, std::vector<T> &hist)
{
    hist.assign(h->hist_len, T{});
    if (!state) return CB_OK;
    const size_t L = h->interp;
    for (size_t k = 0; k < nstate; ++k) {
        const T v = state[k];
        if ((k + 1) % L == 0) {
            const size_t i = (k + 1) / L;  // i-th most recent input sample
            if (i <= h->hist_len) hist[h->hist_len - i] = v;
        } else if (v.x != 0 || v.y != 0) {
            set_error("fir: with interp=%zu the initial state must be zero off the symbol grid (entry %zu)", L, k);
            return CB_ERR_UNSUPPORTED;
        }
    }
    return CB_OK;
}

// chronological input-domain history -> reference state (newest first, nstate entries, zero-stuffed domain)
template <typename Fir, typename T>
static void fir_hist_to_state(const Fir *h, const std::vector<T> &hist, T *state, size_t nstate)
{
    const size_t L = h->interp;
    for (size_t k = 0; k < nstate; ++k) {
        T v{};
        if ((k + 1) % L == 0) {
            const size_t i = (k + 1) / L;
            if (i <= h->hist_len) v = hist[h->hist_len - i];
        }
        state[k] = v;
    }
}
}  // extern "C++"

int cb_fir_create(const float *taps, size_t ntaps, const float *state, size_t nstate, uint32_t decim,
                  uint32_t interp, cb_fir **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(taps || ntaps == 0, CB_ERR_INVALID_ARG, "taps is NULL");
    int rc = ensure_device();
    if (rc) return rc;
    cb_fir *h = new (std::nothrow) cb_fir();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->decim = decim == 0 ? 1 : decim;
    h->interp = interp == 0 ? 1 : interp;
    h->taps.resize(ntaps);
    if (ntaps) memcpy(h->taps.data(), taps, ntaps * sizeof(float2));
    h->nstate = state ? nstate : ntaps;  // None => zeros(len taps)  (fir_node.rs:201-210)
    h->k_eff = (uint32_t)(ntaps < h->nstate ? ntaps : h->nstate);
    h->taps_real = true;
    for (size_t k = 0; k < h->k_eff; ++k)
        if (h->taps[k].y != 0.f) h->taps_real = false;
    const size_t need_in = ceil_div(h->nstate > h->k_eff ? h->nstate : (size_t)h->k_eff, (size_t)h->interp);
    h->hist_len = (uint32_t)round_up(need_in > 128 ? need_in : 128, 2);
    h->cur = 0;
    h->taps_dev = nullptr;
    h->hist[0] = h->hist[1] = nullptr;
    h->stream = nullptr;
    h->tc_img = nullptr;
    h->tc = FirTcPlan{nullptr, 1.f, 0};
    h->qscratch = nullptr;
    h->qscratch_len = 0;
    h->ols_hf = h->ols_twf = h->ols_twi = h->ols_spec = nullptr;
    h->rscratch = nullptr;
    h->rscratch_len = 0;
    h->ols_spec_frames = 0;

    std::vector<float2> hist;
    rc = fir_state_to_hist(h, reinterpret_cast<const float2 *>(state), state ? nstate : 0, hist);
    if (rc) {
        delete h;
        return rc;
    }
#define FIR_TRY(call)                                                    \
    do {                                                                 \
        cudaError_t e__ = (call);                                        \
        if (e__ != cudaSuccess) {                                        \
            cb_fir_destroy(h);                                           \
            return cuda_fail(e__, #call, __FILE__, __LINE__);            \
        }                                                                \
    } while (0)
    FIR_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    if (h->pipe.init(h->stream)) {
        cb_fir_destroy(h);
        return CB_ERR_CUDA;
    }
    FIR_TRY(cudaMalloc(&h->taps_dev, (ntaps ? ntaps : 1) * sizeof(float2)));
    if (ntaps) FIR_TRY(cudaMemcpy(h->taps_dev, h->taps.data(), ntaps * sizeof(float2), cudaMemcpyHostToDevice));
    for (int i = 0; i < 2; ++i) {
        FIR_TRY(cudaMalloc(&h->hist[i], h->hist_len * sizeof(float2)));
        FIR_TRY(cudaMemcpy(h->hist[i], hist.data(), h->hist_len * sizeof(float2), cudaMemcpyHostToDevice));
    }
    // Tensor-core plan (K1-TC).  COMMS_B200_FIR_PATH = auto (default) | cuda | tc selects the kernel
    // family for decim = interp = 1 filters of up to 128 taps; "tc" also drops the batch-size floor.
    {
        const char *path = getenv("COMMS_B200_FIR_PATH");
        const bool want_cuda = path && strcmp(path, "cuda") == 0;
        const bool force_tc = path && strcmp(path, "tc") == 0;
        if (!want_cuda && h->interp == 1 && h->decim == 1 && h->k_eff >= 1 && h->k_eff <= 128) {
            const size_t bytes = fir_tc_image_bytes(h->k_eff);
            std::vector<unsigned char> img(bytes);
            float inv = 1.f;
            fir_tc_build_image(h->taps.data(), h->k_eff, img.data(), &inv);
            FIR_TRY(cudaMalloc(&h->tc_img, bytes));
            FIR_TRY(cudaMemcpy(h->tc_img, img.data(), bytes, cudaMemcpyHostToDevice));
            h->tc = FirTcPlan{h->tc_img, inv, force_tc ? (size_t)1 : ((size_t)1 << 16)};
            h->tc.sample_min = fir_taps_pair_sparse(h->taps.data(), h->k_eff, 1);
        } else if (!want_cuda && h->decim == 1 && h->interp > 1 && fir_ptc_supported(h->k_eff, h->interp, h->taps_real)) {
            // polyphase interpolator on the tensor cores (K3-TC); short banks stay on the CUDA-core
            // polyphase kernel unless forced, long banks (> 16 taps per phase) always use it
            const size_t bytes = fir_ptc_image_bytes(h->k_eff, h->interp, h->taps_real);
            std::vector<unsigned char> img(bytes);
            float inv = 1.f;
            fir_ptc_build_image(h->taps.data(), h->k_eff, h->interp, h->taps_real, img.data(), &inv);
            FIR_TRY(cudaMalloc(&h->tc_img, bytes));
            FIR_TRY(cudaMemcpy(h->tc_img, img.data(), bytes, cudaMemcpyHostToDevice));
            h->tc = FirTcPlan{h->tc_img, inv, force_tc ? (size_t)1 : ((size_t)1 << 16)};
            h->tc.sample_min = fir_taps_pair_sparse(h->taps.data(), h->k_eff, h->interp);
        }
    }
        const char *path2 = getenv("COMMS_B200_FIR_PATH");
        if (!(path2 && strcmp(path2, "cuda") == 0) && h->interp == 1 && h->decim == 1 && h->k_eff > 128 && h->k_eff <= 1025) {
            // long filter: fast convolution.  Hf[k] = sum_t h[t] e^{-2 pi i k t / 4096}, in f64
            std::vector<float2> hf(4096);
            const double w0 = -2.0 * 3.14159265358979323846 / 4096.0;
            for (int k = 0; k < 4096; ++k) {
                double re = 0.0, im = 0.0;
                for (uint32_t t = 0; t < h->k_eff; ++t) {
                    const double ang = w0 * (double)(((long long)k * t) & 4095);
                    const double c = cos(ang), sn = sin(ang);
                    re += (double)h->taps[t].x * c - (double)h->taps[t].y * sn;
                    im += (double)h->taps[t].x * sn + (double)h->taps[t].y * c;
                }
                hf[k] = make_float2((float)re, (float)im);
            }
            FIR_TRY(cudaMalloc(&h->ols_hf, 4096 * sizeof(float2)));
            FIR_TRY(cudaMemcpy(h->ols_hf, hf.data(), 4096 * sizeof(float2), cudaMemcpyHostToDevice));
            for (int inv = 0; inv < 2; ++inv) {
                std::vector<float2> t(fft2_table_len(12));
                fft2_fill_table(12, inv, t.data());
                float2 **dst = inv ? &h->ols_twi : &h->ols_twf;
                FIR_TRY(cudaMalloc(dst, t.size() * sizeof(float2)));
                FIR_TRY(cudaMemcpy(*dst, t.data(), t.size() * sizeof(float2), cudaMemcpyHostToDevice));
            }
        }
#undef FIR_TRY
    *out = h;
    return CB_OK;
}

int cb_fir_destroy(cb_fir *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    if (h->taps_dev) cudaFree(h->taps_dev);
    if (h->tc_img) cudaFree(h->tc_img);
    for (int i = 0; i < 2; ++i)
        if (h->fix[i].dev) cudaFree(h->fix[i].dev);
    if (h->qscratch) cudaFree(h->qscratch);
    if (h->rscratch) cudaFree(h->rscratch);
    if (h->ols_hf) cudaFree(h->ols_hf);
    if (h->ols_twf) cudaFree(h->ols_twf);
    if (h->ols_twi) cudaFree(h->ols_twi);
    if (h->ols_spec) cudaFree(h->ols_spec);
    for (int i = 0; i < 2; ++i)
        if (h->hist[i]) cudaFree(h->hist[i]);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_fir_out_len(const cb_fir *h, size_t n_in, size_t *n_out)
{
    CB_REQUIRE(h && n_out, CB_ERR_INVALID_ARG, "NULL argument");
    *n_out = fir_out_len(h, n_in);
    return CB_OK;
}

void *cb_fir_stream(cb_fir *h) { return h ? (void *)h->stream : nullptr; }

// the lane's fix-up list, grown to hold every tile a launch over n inputs could flag (NULL when it cannot be allocated:
// the launch then runs without the fall-back pass, as before)
static FirFix *fir_fix_for(cb_fir *h, size_t n, int lane)
{
    if (!h->tc_img) return nullptr;
    FirFix &f = h->fix[lane & 1];
    const size_t need = fir_fix_tiles(n);
    if (f.cap < need) {
        if (f.dev) cudaFree(f.dev);  // waits for launches that still use it
        f.dev = nullptr;
        f.cap = 0;
        f.calls = 0;
        const size_t cap = need < 4096 ? 4096 : need * 2;
        // (the memset runs on the legacy default stream, which non-blocking streams do not wait for: make sure it has
        // landed before a kernel on the caller's stream reads the counters -- this happens once per handle and growth)
        if (cudaMalloc(&f.dev, (cap + 2) * sizeof(unsigned)) != cudaSuccess || cudaMemset(f.dev, 0, 2 * sizeof(unsigned)) != cudaSuccess ||
            cudaStreamSynchronize(cudaStreamLegacy) != cudaSuccess) {
            (void)cudaGetLastError();
            if (f.dev) cudaFree(f.dev);
            f.dev = nullptr;
            return nullptr;
        }
        f.cap = (unsigned)cap;
    }
    return &f;
}

static int fir_launch_segment(cb_fir *h, const float2 *x, size_t n, const float2 *hist_in, float2 *hist_out,
                              float2 *y, cudaStream_t s, int lane = 0)
{
    h->tc.fix = fir_fix_for(h, n, lane);
    // long filters and long batches: overlap-save fast convolution (spectra scratch grown on demand; when it
    // cannot be allocated the direct-form kernel below is used)
    // COMMS_B200_FIR_OLS=split: the two-kernel form with the spectra in a scratch (kept for comparison); default: one
    // fused kernel per frame, no scratch
    static const bool ols_split = [] { const char *e = getenv("COMMS_B200_FIR_OLS"); return e && strcmp(e, "split") == 0; }();
    if (h->ols_hf != nullptr && n >= 8192 && !ols_split)
        return launch_fir_ols(x, n, hist_in, hist_out, h->hist_len, h->k_eff, h->ols_hf, h->ols_twf, h->ols_twi, nullptr, y, s);
    if (h->ols_hf != nullptr && n >= 8192) {
        const size_t frames = fir_ols_frames(n, h->k_eff);
        if (h->ols_spec_frames < frames) {
            if (h->ols_spec) cudaFree(h->ols_spec);
            h->ols_spec = nullptr;
            h->ols_spec_frames = 0;
            if (cudaMalloc(&h->ols_spec, frames * 4096 * sizeof(float2)) == cudaSuccess) h->ols_spec_frames = frames;
            else cudaGetLastError();
        }
        if (h->ols_spec_frames >= frames)
            return launch_fir_ols(x, n, hist_in, hist_out, h->hist_len, h->k_eff, h->ols_hf, h->ols_twf, h->ols_twi,
                                  h->ols_spec, y, s);
    }
    // k_eff == 0 (zip over an empty state, fir.rs:99) runs as an all-zero filter: outputs are 0
    FirSeg seg{x, hist_in, hist_out, y, n, fir_out_len(h, n), h->hist_len, h->k_eff, h->interp, h->decim};
    return launch_fir(seg, h->taps_dev, h->taps.data(), h->taps_real, h->tc_img ? &h->tc : nullptr, s);
}

int cb_fir_run_dev(cb_fir *h, const float *d_in, size_t n_in, float *d_out, size_t out_cap, size_t *n_out,
                   void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_NO_ALIAS(d_in, n_in * sizeof(float2), d_out, no * sizeof(float2), "fir");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);
    if (rc) return rc;
    rc = fir_launch_segment(h, reinterpret_cast<const float2 *>(d_in), n_in, h->hist[h->cur], h->hist[h->cur ^ 1],
                            reinterpret_cast<float2 *>(d_out), s);
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

int cb_fir_run_dev_i16(cb_fir *h, const float *d_in, size_t n_in, float scale, int16_t *d_out, size_t out_cap,
                       size_t *n_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_NO_ALIAS(d_in, n_in * sizeof(float2), d_out, no * 2 * sizeof(int16_t), "fir");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    FirSeg seg{reinterpret_cast<const float2 *>(d_in), h->hist[h->cur], h->hist[h->cur ^ 1], nullptr, n_in, no,
               h->hist_len, h->k_eff, h->interp, h->decim};
    seg.y16 = d_out;
    seg.qscale = scale;
    seg.y = reinterpret_cast<float2 *>(d_out);  // unused by the fused kernel (alignment checks only)
    int rc = h->last.begin(s);
    if (rc) return rc;
    h->tc.fix = fir_fix_for(h, n_in, 0);
    if (fir_fuses_i16(seg, h->taps_real, h->tc_img ? &h->tc : nullptr)) {
        rc = launch_fir(seg, h->taps_dev, h->taps.data(), h->taps_real, &h->tc, s);
    } else {  // filter into an f32 scratch, then the stand-alone quantiser
        if (h->qscratch_len < no) {
            if (h->qscratch) CB_CUDA(cudaFree(h->qscratch));
            h->qscratch = nullptr;
            h->qscratch_len = 0;
            CB_CUDA(cudaMalloc(&h->qscratch, no * sizeof(float2)));
            h->qscratch_len = no;
        }
        seg.y16 = nullptr;
        seg.y = h->qscratch;
        rc = launch_fir(seg, h->taps_dev, h->taps.data(), h->taps_real, h->tc_img ? &h->tc : nullptr, s);
        if (rc == CB_OK) rc = launch_quantize_i16(reinterpret_cast<const float *>(h->qscratch), d_out, 2 * no, scale, s);
    }
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

// Real samples in, real parts out: the Convert2Node -> BatchFirNode -> Convert3Node [-> DecimateNode] run of
// examples/fm_radio.rs:98-164.  One fused kernel for <= 64 taps and D in {2, 4, 5, 8, 10}; any other shape widens into a
// scratch, runs the complex filter and takes the real parts.  The carried state stays the handle's complex history.
int cb_fir_run_real_dev(cb_fir *h, const float *d_in, size_t n_in, float *d_out, size_t out_cap, size_t *n_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_NO_ALIAS(d_in, n_in * sizeof(float), d_out, no * sizeof(float), "fir");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);
    if (rc) return rc;
    if (fir_real_applicable(h->k_eff, h->interp, h->decim) && h->hist_len >= h->k_eff) {
        rc = launch_fir_real(d_in, n_in, h->hist[h->cur], h->hist[h->cur ^ 1], h->hist_len, h->taps.data(), h->k_eff,
                             h->decim, d_out, s);
    } else {
        if (h->rscratch_len < n_in + no) {
            if (h->rscratch) CB_CUDA(cudaFree(h->rscratch));
            h->rscratch = nullptr;
            h->rscratch_len = 0;
            CB_CUDA(cudaMalloc(&h->rscratch, (n_in + no) * sizeof(float2)));
            h->rscratch_len = n_in + no;
        }
        float2 *wide = h->rscratch, *res = h->rscratch + n_in;
        rc = launch_real_to_complex(d_in, wide, n_in, s);
        if (rc == CB_OK) rc = fir_launch_segment(h, wide, n_in, h->hist[h->cur], h->hist[h->cur ^ 1], res, s);
        if (rc == CB_OK) rc = launch_complex_real(res, d_out, no, s);
    }
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

int cb_fir_run_real(cb_fir *h, const float *in, size_t n_in, float *out, size_t out_cap, size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    int rc = h->pipe.reserve(n_in * sizeof(float), no * sizeof(float));
    if (rc) return rc;
    cudaStream_t s = h->pipe.lane[0];
    CB_CUDA(cudaMemcpyAsync(h->pipe.in[0], in, n_in * sizeof(float), cudaMemcpyHostToDevice, s));
    rc = cb_fir_run_real_dev(h, reinterpret_cast<const float *>(h->pipe.in[0]), n_in, reinterpret_cast<float *>(h->pipe.out[0]),
                             no, nullptr, s);
    if (rc) return rc;
    CB_CUDA(cudaMemcpyAsync(out, h->pipe.out[0], no * sizeof(float), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
    return CB_OK;
}

int cb_fir_run_i16(cb_fir *h, const float *in, size_t n_in, float scale, int16_t *out, size_t out_cap, size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    int rc = h->pipe.reserve(n_in * sizeof(float2), no * 2 * sizeof(int16_t));
    if (rc) return rc;
    cudaStream_t s = h->pipe.lane[0];
    CB_CUDA(cudaMemcpyAsync(h->pipe.in[0], in, n_in * sizeof(float2), cudaMemcpyHostToDevice, s));
    rc = cb_fir_run_dev_i16(h, reinterpret_cast<const float *>(h->pipe.in[0]), n_in, scale,
                            reinterpret_cast<int16_t *>(h->pipe.out[0]), no, nullptr, s);
    if (rc) return rc;
    CB_CUDA(cudaMemcpyAsync(out, h->pipe.out[0], no * 2 * sizeof(int16_t), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
    return CB_OK;
}

int cb_fir_run(cb_fir *h, const float *in, size_t n_in, float *out, size_t out_cap, size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    const float2 *hin = reinterpret_cast<const float2 *>(in);
    float2 *hout = reinterpret_cast<float2 *>(out);
    const size_t H = h->hist_len;
    // chunk starts must keep the decimation grid: multiples of D input samples
    size_t chunk = HOST_CHUNK / h->decim * h->decim;
    if (chunk < 4 * H || n_in <= chunk) chunk = n_in;
    int rc = h->last.sync();  // a *_run_dev on a caller's stream may still be using the carried state
    if (rc) return rc;
    rc = h->pipe.reserve((chunk + H) * sizeof(float2), fir_out_len(h, chunk) * sizeof(float2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n_in * sizeof(float2), (chunk + H) * sizeof(float2), out, no * sizeof(float2),
                            fir_out_len(h, chunk) * sizeof(float2));
    if (rc) return rc;
    // Small messages (what the reference's graphs pass around: a 4096-symbol message is 32 KiB in, 128 KiB out): no
    // copy engine at all -- the kernel reads the samples from, and writes the result to, pinned host memory (the
    // caller's own when it is pinned, the handle's slots around a memcpy when it is pageable), one launch and one wait.
    // Only the CUDA-core kernels take this path (plain loads and stores); history and carried state stay on the device.
    if (chunk == n_in && (n_in + no) * sizeof(float2) <= ZEROCOPY_MAX_BYTES && !(h->tc_img && n_in >= h->tc.min_samples) &&
        !(h->ols_hf != nullptr && n_in >= 8192) && !ranges_overlap(hin, n_in * sizeof(float2), hout, no * sizeof(float2))) {
        const float2 *dx = h->pipe.stage_in ? nullptr : host_device_view(hin);
        float2 *dy = h->pipe.stage_out ? nullptr : const_cast<float2 *>(host_device_view(hout));
        const bool copy_in = dx == nullptr, copy_out = dy == nullptr;
        if ((!copy_in || h->pipe.stage_in) && (!copy_out || h->pipe.stage_out)) {
            if (copy_in) {
                memcpy(h->pipe.pin_in[0], hin, n_in * sizeof(float2));
                dx = reinterpret_cast<const float2 *>(h->pipe.pin_in[0]);
            }
            if (copy_out) dy = reinterpret_cast<float2 *>(h->pipe.pin_out[0]);
            rc = fir_launch_segment(h, dx, n_in, h->hist[h->cur], h->hist[h->cur ^ 1], dy, h->pipe.lane[0], 0);
            if (rc) return rc;
            CB_CUDA(cudaStreamSynchronize(h->pipe.lane[0]));
            if (copy_out) memcpy(hout, h->pipe.pin_out[0], no * sizeof(float2));
            h->cur ^= 1;
            return CB_OK;
        }
    }
    size_t done = 0, out_done = 0;
    for (int i = 0; done < n_in; ++i) {
        const int l = i & 1;
        const size_t n = n_in - done < chunk ? n_in - done : chunk;
        const bool last = done + n == n_in;
        cudaStream_t s = h->pipe.lane[l];
        float2 *slot = reinterpret_cast<float2 *>(h->pipe.in[l]);
        const float2 *hist_in;
        if (done == 0) {
            hist_in = h->hist[h->cur];
            rc = h->pipe.h2d(l, slot + H, hin, n * sizeof(float2));
        } else {  // the halo is the tail of the previous chunk, re-sent with this one
            hist_in = slot;
            rc = h->pipe.h2d(l, slot, hin + done - H, (n + H) * sizeof(float2));
        }
        if (rc) return rc;
        float2 *y = reinterpret_cast<float2 *>(h->pipe.out[l]);
        rc = fir_launch_segment(h, slot + H, n, hist_in, last ? h->hist[h->cur ^ 1] : nullptr, y, s, l);
        if (rc) return rc;
        const size_t m = fir_out_len(h, n);
        rc = h->pipe.d2h(l, hout + out_done, y, m * sizeof(float2));
        if (rc) return rc;
        done += n;
        out_done += m;
    }
    rc = h->pipe.sync();
    if (rc) return rc;
    h->cur ^= 1;
    return CB_OK;
}

// ---- i16 IQ on both edges (src/io/raw_iq.rs:78-140 IQBatchInput, :185-223 IQBatchOutput): x = in_scale * (i16 as f32),
// the handle's filter, y16 = (out_scale * y) as i16.  Half the bytes of the f32 entries on every edge.
// One filter step with f32 input already on the device -> i16 output (fused epilogue for the tensor-core polyphase banks).
static int fir_segment_to_i16(cb_fir *h, const float2 *x, size_t n, const float2 *hist_in, float2 *hist_out, float out_scale,
                              int16_t *y16, float2 *yscratch, cudaStream_t s, int lane)
{
    const size_t no = fir_out_len(h, n);
    h->tc.fix = fir_fix_for(h, n, lane);
    FirSeg seg{x, hist_in, hist_out, nullptr, n, no, h->hist_len, h->k_eff, h->interp, h->decim};
    seg.y16 = y16;
    seg.qscale = out_scale;
    seg.y = reinterpret_cast<float2 *>(y16);
    if (fir_fuses_i16(seg, h->taps_real, h->tc_img ? &h->tc : nullptr))
        return launch_fir(seg, h->taps_dev, h->taps.data(), h->taps_real, &h->tc, s);
    int rc = fir_launch_segment(h, x, n, hist_in, hist_out, yscratch, s, lane);
    if (rc) return rc;
    return launch_quantize_i16(reinterpret_cast<const float *>(yscratch), y16, 2 * no, out_scale, s);
}

// Plain filters of up to 128 taps on a long enough batch: the tensor-core kernel reads the i16 IQ words itself and its
// epilogue writes i16 IQ words (fir_tc_kernel.cu, IQ16) -- 4 + 4 bytes per sample, one launch.
static bool fir_iq16_fused(const cb_fir *h, size_t n, const int16_t *x16, const int16_t *y16)
{
    if (!h->tc_img || n < h->tc.min_samples || h->interp != 1 || h->decim != 1 || h->k_eff == 0) return false;
    if (const char *e = getenv("COMMS_B200_FIR_IQ16"))  // "split": cast, filter and quantiser as separate passes (for comparison)
        if (strcmp(e, "split") == 0) return false;
    FirSeg seg{nullptr, h->hist[0], nullptr, nullptr, n, n, h->hist_len, h->k_eff, h->interp, h->decim};
    return fir_tc_iq16_applicable(seg, x16, y16);
}

int cb_fir_run_dev_iq16(cb_fir *h, const int16_t *d_in, size_t n_in, float in_scale, float out_scale, int16_t *d_out,
                        size_t out_cap, size_t *n_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_NO_ALIAS(d_in, n_in * 2 * sizeof(int16_t), d_out, no * 2 * sizeof(int16_t), "fir");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);
    if (rc) return rc;
    if (fir_iq16_fused(h, n_in, d_in, d_out)) {
        FirSeg seg{nullptr, h->hist[h->cur], h->hist[h->cur ^ 1], nullptr, n_in, no, h->hist_len, h->k_eff, h->interp, h->decim};
        h->tc.fix = fir_fix_for(h, n_in, 0);
        rc = launch_fir_tc_iq16(seg, d_in, in_scale, d_out, out_scale, h->tc, h->taps_dev, s);
        if (rc) return rc;
        h->cur ^= 1;
        return h->last.end(s);
    }
    const size_t res_off = round_up(n_in, (size_t)4);  // the f32 result 32-byte aligned like the input (tensor-core path)
    if (h->rscratch_len < res_off + no) {  // widened input followed by the f32 result
        if (h->rscratch) CB_CUDA(cudaFree(h->rscratch));
        h->rscratch = nullptr;
        h->rscratch_len = 0;
        CB_CUDA(cudaMalloc(&h->rscratch, (res_off + no) * sizeof(float2)));
        h->rscratch_len = res_off + no;
    }
    float2 *wide = h->rscratch, *res = h->rscratch + res_off;
    rc = launch_convert_i16(d_in, reinterpret_cast<float *>(wide), 2 * n_in, in_scale, s);
    if (rc == CB_OK)
        rc = fir_segment_to_i16(h, wide, n_in, h->hist[h->cur], h->hist[h->cur ^ 1], out_scale, d_out, res, s, 0);
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

int cb_fir_run_iq16(cb_fir *h, const int16_t *in, size_t n_in, float in_scale, float out_scale, int16_t *out, size_t out_cap,
                    size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir: out_cap %zu < %zu outputs", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    const size_t H = h->hist_len, IQ = 2 * sizeof(int16_t);
    size_t chunk = HOST_CHUNK * 2 / h->decim * h->decim;  // twice the samples of an f32 chunk: the same 32 MiB per copy
    if (chunk < 4 * H || n_in <= chunk) chunk = n_in;
    const size_t chunk_out = fir_out_len(h, chunk);
    int rc = h->last.sync();
    if (rc) return rc;
    rc = h->pipe.reserve((chunk + H) * IQ, chunk_out * IQ);
    if (rc) return rc;
    rc = h->pipe.reserve_aux((chunk + H) * sizeof(float2), chunk_out * sizeof(float2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n_in * IQ, (chunk + H) * IQ, out, no * IQ, chunk_out * IQ);
    if (rc) return rc;
    const char *hin = reinterpret_cast<const char *>(in);
    char *hout = reinterpret_cast<char *>(out);
    size_t done = 0, out_done = 0;
    for (int i = 0; done < n_in; ++i) {
        const int l = i & 1;
        const size_t n = n_in - done < chunk ? n_in - done : chunk;
        const bool last = done + n == n_in;
        cudaStream_t s = h->pipe.lane[l];
        char *slot16 = reinterpret_cast<char *>(h->pipe.in[l]);
        float2 *wide = reinterpret_cast<float2 *>(h->pipe.aux_in[l]);
        const float2 *hist_in;
        if (fir_iq16_fused(h, n, reinterpret_cast<const int16_t *>(slot16 + H * IQ), reinterpret_cast<const int16_t *>(h->pipe.out[l]))) {
            // the kernel reads and writes the i16 words itself; only a later chunk's halo (the tail of the previous
            // chunk, re-sent with this one) is widened, because the kernel takes its history as f32
            if (done == 0) {
                hist_in = h->hist[h->cur];
                rc = h->pipe.h2d(l, slot16 + H * IQ, hin, n * IQ);
            } else {
                hist_in = wide;
                rc = h->pipe.h2d(l, slot16, hin + (done - H) * IQ, (n + H) * IQ);
                if (rc == CB_OK) rc = launch_convert_i16(reinterpret_cast<const int16_t *>(slot16), reinterpret_cast<float *>(wide), 2 * H, in_scale, s);
            }
            if (rc) return rc;
            int16_t *y16 = reinterpret_cast<int16_t *>(h->pipe.out[l]);
            FirSeg seg{nullptr, hist_in, last ? h->hist[h->cur ^ 1] : nullptr, nullptr, n, n, h->hist_len, h->k_eff, h->interp, h->decim};
            h->tc.fix = fir_fix_for(h, n, l);
            rc = launch_fir_tc_iq16(seg, reinterpret_cast<const int16_t *>(slot16 + H * IQ), in_scale, y16, out_scale, h->tc,
                                    h->taps_dev, s);
            if (rc) return rc;
            rc = h->pipe.d2h(l, hout + out_done * IQ, y16, n * IQ);
            if (rc) return rc;
            done += n;
            out_done += n;
            continue;
        }
        if (done == 0) {  // the carried history is already f32
            hist_in = h->hist[h->cur];
            rc = h->pipe.h2d(l, slot16 + H * IQ, hin, n * IQ);
            if (rc == CB_OK) rc = launch_convert_i16(reinterpret_cast<const int16_t *>(slot16 + H * IQ), reinterpret_cast<float *>(wide + H), 2 * n, in_scale, s);
        } else {  // the halo is the tail of the previous chunk, re-sent (and re-converted) with this one
            hist_in = wide;
            rc = h->pipe.h2d(l, slot16, hin + (done - H) * IQ, (n + H) * IQ);
            if (rc == CB_OK) rc = launch_convert_i16(reinterpret_cast<const int16_t *>(slot16), reinterpret_cast<float *>(wide), 2 * (n + H), in_scale, s);
        }
        if (rc) return rc;
        int16_t *y16 = reinterpret_cast<int16_t *>(h->pipe.out[l]);
        rc = fir_segment_to_i16(h, wide + H, n, hist_in, last ? h->hist[h->cur ^ 1] : nullptr, out_scale, y16,
                                reinterpret_cast<float2 *>(h->pipe.aux_out[l]), s, l);
        if (rc) return rc;
        const size_t m = fir_out_len(h, n);
        rc = h->pipe.d2h(l, hout + out_done * IQ, y16, m * IQ);
        if (rc) return rc;
        done += n;
        out_done += m;
    }
    rc = h->pipe.sync();
    if (rc) return rc;
    h->cur ^= 1;
    return CB_OK;
}

int cb_fir_state_len(const cb_fir *h, size_t *nstate)
{
    CB_REQUIRE(h && nstate, CB_ERR_INVALID_ARG, "NULL argument");
    *nstate = h->nstate;
    return CB_OK;
}

int cb_fir_get_state(cb_fir *h, float *state, size_t nstate)
{
    CB_REQUIRE(h && (state || nstate == 0), CB_ERR_INVALID_ARG, "NULL argument");
    CB_REQUIRE(nstate == h->nstate, CB_ERR_SIZE, "fir: state length %zu != %zu", nstate, h->nstate);
    CB_CUDA(cudaSetDevice(h->device));
    CB_CUDA(cudaStreamSynchronize(h->stream));
    {
        const int rcl = h->last.sync();
        if (rcl) return rcl;
    }
    std::vector<float2> hist(h->hist_len);
    CB_CUDA(cudaMemcpy(hist.data(), h->hist[h->cur], h->hist_len * sizeof(float2), cudaMemcpyDeviceToHost));
    fir_hist_to_state(h, hist, reinterpret_cast<float2 *>(state), nstate);
    return CB_OK;
}

int cb_fir_set_state(cb_fir *h, const float *state, size_t nstate)
{
    CB_REQUIRE(h && state, CB_ERR_INVALID_ARG, "NULL argument");
    CB_REQUIRE(nstate == h->nstate, CB_ERR_SIZE, "fir: state length %zu != %zu", nstate, h->nstate);
    CB_CUDA(cudaSetDevice(h->device));
    std::vector<float2> hist;
    int rc = fir_state_to_hist(h, reinterpret_cast<const float2 *>(state), nstate, hist);
    if (rc) return rc;
    CB_CUDA(cudaStreamSynchronize(h->stream));
    rc = h->last.sync();
    if (rc) return rc;
    CB_CUDA(cudaMemcpy(h->hist[h->cur], hist.data(), h->hist_len * sizeof(float2), cudaMemcpyHostToDevice));
    return CB_OK;
}

// ============================================================================ FIR over Complex<f64>
// The same filter, state and resampling semantics as cb_fir, over double2 samples, with one direct-form kernel family
// (fir_f64_kernels.cu) whose per-output FMA chain is fixed: no tensor-core, overlap-save or zero-copy paths.
struct cb_fir_f64 {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    double2 *taps_dev;
    size_t nstate;      // reference state length (zero-stuffed domain when interp > 1)
    uint32_t k_eff;     // min(ntaps, nstate)
    bool taps_real;
    uint32_t decim, interp;
    uint32_t hist_len;  // input-domain samples kept
    double2 *hist[2];
    int cur;
    LastUse last;
};

int cb_fir_f64_create(const double *taps, size_t ntaps, const double *state, size_t nstate, uint32_t decim,
                      uint32_t interp, cb_fir_f64 **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(taps || ntaps == 0, CB_ERR_INVALID_ARG, "taps is NULL");
    // the kernels skip the products with stuffed zeros and padding, so a non-finite tap could not poison the outputs
    // the way the reference's fold over the zero-stuffed stream does: reject it instead
    for (size_t k = 0; k < 2 * ntaps; ++k)
        CB_REQUIRE(std::isfinite(taps[k]), CB_ERR_INVALID_ARG, "fir_f64: tap %zu is not finite", k / 2);
    int rc = ensure_device();
    if (rc) return rc;
    cb_fir_f64 *h = new (std::nothrow) cb_fir_f64();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->decim = decim == 0 ? 1 : decim;
    h->interp = interp == 0 ? 1 : interp;
    h->nstate = state ? nstate : ntaps;  // None => zeros(len taps)  (fir_node.rs:201-210)
    h->k_eff = (uint32_t)(ntaps < h->nstate ? ntaps : h->nstate);
    h->taps_real = true;
    for (size_t k = 0; k < h->k_eff; ++k)
        if (taps[2 * k + 1] != 0.0) h->taps_real = false;
    const size_t need_in = ceil_div(h->nstate > h->k_eff ? h->nstate : (size_t)h->k_eff, (size_t)h->interp);
    h->hist_len = (uint32_t)(need_in > 1 ? need_in : 1);
    h->cur = 0;
    h->taps_dev = nullptr;
    h->hist[0] = h->hist[1] = nullptr;
    h->stream = nullptr;
    std::vector<double2> hist;
    rc = fir_state_to_hist(h, reinterpret_cast<const double2 *>(state), state ? nstate : 0, hist);
    if (rc) {
        delete h;
        return rc;
    }
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess && h->pipe.init(h->stream)) e = cudaErrorUnknown;
    if (e == cudaSuccess) e = cudaMalloc(&h->taps_dev, (ntaps ? ntaps : 1) * sizeof(double2));
    if (e == cudaSuccess && ntaps) e = cudaMemcpy(h->taps_dev, taps, ntaps * sizeof(double2), cudaMemcpyHostToDevice);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaMalloc(&h->hist[i], h->hist_len * sizeof(double2));
        if (e == cudaSuccess) e = cudaMemcpy(h->hist[i], hist.data(), h->hist_len * sizeof(double2), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        cb_fir_f64_destroy(h);
        return cuda_fail(e, "fir_f64 create", __FILE__, __LINE__);
    }
    *out = h;
    return CB_OK;
}

int cb_fir_f64_destroy(cb_fir_f64 *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    if (h->taps_dev) cudaFree(h->taps_dev);
    for (int i = 0; i < 2; ++i)
        if (h->hist[i]) cudaFree(h->hist[i]);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_fir_f64_out_len(const cb_fir_f64 *h, size_t n_in, size_t *n_out)
{
    CB_REQUIRE(h && n_out, CB_ERR_INVALID_ARG, "NULL argument");
    *n_out = fir_out_len(h, n_in);
    return CB_OK;
}

void *cb_fir_f64_stream(cb_fir_f64 *h) { return h ? (void *)h->stream : nullptr; }

static int fir64_launch(cb_fir_f64 *h, const double2 *x, size_t n, const double2 *hist_in, double2 *hist_out, double2 *y,
                        cudaStream_t s)
{
    const Fir64Seg seg{x, hist_in, hist_out, y, n, fir_out_len(h, n), h->hist_len, h->k_eff, h->interp, h->decim};
    return launch_fir_f64(seg, h->taps_dev, h->taps_real, s);
}

int cb_fir_f64_run_dev(cb_fir_f64 *h, const double *d_in, size_t n_in, double *d_out, size_t out_cap, size_t *n_out,
                       void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(((reinterpret_cast<uintptr_t>(d_in) | reinterpret_cast<uintptr_t>(d_out)) & 15) == 0, CB_ERR_INVALID_ARG,
               "fir_f64: d_in and d_out must be 16-byte aligned");  // read and written as double2
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir_f64: out_cap %zu < %zu outputs", out_cap, no);
    CB_NO_ALIAS(d_in, n_in * sizeof(double2), d_out, no * sizeof(double2), "fir_f64");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);
    if (rc) return rc;
    rc = fir64_launch(h, reinterpret_cast<const double2 *>(d_in), n_in, h->hist[h->cur], h->hist[h->cur ^ 1],
                      reinterpret_cast<double2 *>(d_out), s);
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

// Host Vec in / Vec out: chunks of HOST_CHUNK samples pipelined over the handle's two lanes (H2D, filter, D2H); each
// chunk after the first re-sends the previous chunk's last hist_len samples as its history.
int cb_fir_f64_run(cb_fir_f64 *h, const double *in, size_t n_in, double *out, size_t out_cap, size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = fir_out_len(h, n_in);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "fir_f64: out_cap %zu < %zu outputs", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    const double2 *hin = reinterpret_cast<const double2 *>(in);
    double2 *hout = reinterpret_cast<double2 *>(out);
    const size_t H = h->hist_len;
    size_t chunk = HOST_CHUNK / h->decim * h->decim;  // chunk starts keep the decimation grid
    if (chunk < 4 * H || n_in <= chunk) chunk = n_in;
    const size_t chunk_out = fir_out_len(h, chunk);
    int rc = h->last.sync();  // a *_run_dev on a caller's stream may still be using the carried state
    if (rc) return rc;
    rc = h->pipe.reserve((chunk + H) * sizeof(double2), chunk_out * sizeof(double2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n_in * sizeof(double2), (chunk + H) * sizeof(double2), out, no * sizeof(double2),
                            chunk_out * sizeof(double2));
    if (rc) return rc;
    size_t done = 0, out_done = 0;
    for (int i = 0; done < n_in; ++i) {
        const int l = i & 1;
        const size_t n = n_in - done < chunk ? n_in - done : chunk;
        const bool last = done + n == n_in;
        cudaStream_t s = h->pipe.lane[l];
        double2 *slot = reinterpret_cast<double2 *>(h->pipe.in[l]);
        const double2 *hist_in;
        if (done == 0) {
            hist_in = h->hist[h->cur];
            rc = h->pipe.h2d(l, slot + H, hin, n * sizeof(double2));
        } else {
            hist_in = slot;
            rc = h->pipe.h2d(l, slot, hin + done - H, (n + H) * sizeof(double2));
        }
        if (rc) return rc;
        double2 *y = reinterpret_cast<double2 *>(h->pipe.out[l]);
        rc = fir64_launch(h, slot + H, n, hist_in, last ? h->hist[h->cur ^ 1] : nullptr, y, s);
        if (rc) return rc;
        const size_t m = fir_out_len(h, n);
        rc = h->pipe.d2h(l, hout + out_done, y, m * sizeof(double2));
        if (rc) return rc;
        done += n;
        out_done += m;
    }
    rc = h->pipe.sync();
    if (rc) return rc;
    h->cur ^= 1;
    return CB_OK;
}

int cb_fir_f64_state_len(const cb_fir_f64 *h, size_t *nstate)
{
    CB_REQUIRE(h && nstate, CB_ERR_INVALID_ARG, "NULL argument");
    *nstate = h->nstate;
    return CB_OK;
}

int cb_fir_f64_get_state(cb_fir_f64 *h, double *state, size_t nstate)
{
    CB_REQUIRE(h && (state || nstate == 0), CB_ERR_INVALID_ARG, "NULL argument");
    CB_REQUIRE(nstate == h->nstate, CB_ERR_SIZE, "fir_f64: state length %zu != %zu", nstate, h->nstate);
    CB_CUDA(cudaSetDevice(h->device));
    CB_CUDA(cudaStreamSynchronize(h->stream));
    int rc = h->last.sync();
    if (rc) return rc;
    std::vector<double2> hist(h->hist_len);
    CB_CUDA(cudaMemcpy(hist.data(), h->hist[h->cur], h->hist_len * sizeof(double2), cudaMemcpyDeviceToHost));
    fir_hist_to_state(h, hist, reinterpret_cast<double2 *>(state), nstate);
    return CB_OK;
}

int cb_fir_f64_set_state(cb_fir_f64 *h, const double *state, size_t nstate)
{
    CB_REQUIRE(h && state, CB_ERR_INVALID_ARG, "NULL argument");
    CB_REQUIRE(nstate == h->nstate, CB_ERR_SIZE, "fir_f64: state length %zu != %zu", nstate, h->nstate);
    CB_CUDA(cudaSetDevice(h->device));
    std::vector<double2> hist;
    int rc = fir_state_to_hist(h, reinterpret_cast<const double2 *>(state), nstate, hist);
    if (rc) return rc;
    CB_CUDA(cudaStreamSynchronize(h->stream));
    rc = h->last.sync();
    if (rc) return rc;
    CB_CUDA(cudaMemcpy(h->hist[h->cur], hist.data(), h->hist_len * sizeof(double2), cudaMemcpyHostToDevice));
    return CB_OK;
}

// ============================================================================ resample
static size_t decim_len(size_t n, size_t rate) { return rate <= 1 ? n : ceil_div(n, rate); }
static size_t ups_len(size_t n, size_t rate) { return rate <= 1 ? n : n * rate; }

int cb_decimate_dev(const void *d_in, size_t n, size_t elem, size_t rate, void *d_out, size_t out_cap, size_t *n_out,
                    void *stream)
{
    const size_t m = decim_len(n, rate);
    if (n_out) *n_out = m;
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= m, CB_ERR_SIZE, "decimate: out_cap %zu < %zu", out_cap, m);
    int rc = ensure_device();
    if (rc) return rc;
    if (rate <= 1) {
        CB_CUDA(cudaMemcpyAsync(d_out, d_in, n * elem, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        return CB_OK;
    }
    return launch_decimate(d_in, d_out, m, elem, rate, (cudaStream_t)stream);
}

int cb_upsample_dev(const void *d_in, size_t n, size_t elem, size_t rate, void *d_out, size_t out_cap, size_t *n_out,
                    void *stream)
{
    const size_t m = ups_len(n, rate);
    if (n_out) *n_out = m;
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= m, CB_ERR_SIZE, "upsample: out_cap %zu < %zu", out_cap, m);
    int rc = ensure_device();
    if (rc) return rc;
    if (rate <= 1) {
        CB_CUDA(cudaMemcpyAsync(d_out, d_in, n * elem, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        return CB_OK;
    }
    return launch_upsample(d_in, d_out, m, elem, rate, (cudaStream_t)stream);
}

static int resample_host(bool up, const void *in, size_t n, size_t elem, size_t rate, void *out, size_t out_cap,
                         size_t *n_out)
{
    const size_t m = up ? ups_len(n, rate) : decim_len(n, rate);
    if (n_out) *n_out = m;
    if (n == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= m, CB_ERR_SIZE, "resample: out_cap %zu < %zu", out_cap, m);
    int rc = ensure_device();
    if (rc) return rc;
    void *din = nullptr, *dout = nullptr;
    CB_CUDA(cudaMalloc(&din, n * elem));
    cudaError_t e = cudaMalloc(&dout, m * elem);
    if (e != cudaSuccess) {
        cudaFree(din);
        return cuda_fail(e, "cudaMalloc", __FILE__, __LINE__);
    }
    rc = CB_OK;
    e = cudaMemcpy(din, in, n * elem, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        size_t mm;
        rc = up ? cb_upsample_dev(din, n, elem, rate, dout, m, &mm, nullptr)
                : cb_decimate_dev(din, n, elem, rate, dout, m, &mm, nullptr);
        if (rc == CB_OK) e = cudaMemcpy(out, dout, m * elem, cudaMemcpyDeviceToHost);
    }
    cudaFree(din);
    cudaFree(dout);
    if (e != cudaSuccess) return cuda_fail(e, "resample copy", __FILE__, __LINE__);
    return rc;
}

int cb_decimate(const void *in, size_t n, size_t elem, size_t rate, void *out, size_t out_cap, size_t *n_out)
{
    return resample_host(false, in, n, elem, rate, out, out_cap, n_out);
}

int cb_upsample(const void *in, size_t n, size_t elem, size_t rate, void *out, size_t out_cap, size_t *n_out)
{
    return resample_host(true, in, n, elem, rate, out, out_cap, n_out);
}

// ============================================================================ mixer
static double wrap_dphase(double d)  // Mixer::new (src/mixer.rs:43-51)
{
    const double twopi = 2.0 * M_PI;
    if (!std::isfinite(d)) return d;
    while (d >= twopi) d -= twopi;
    while (d < 0.0) d += twopi;
    return d;
}

static double advance_phase(double phase, double dphase, size_t n)
{
    const long double twopi = 6.283185307179586476925286766559L;
    long double p = (long double)phase + (long double)n * (long double)dphase;
    p = fmodl(p, twopi);
    if (p < 0) p += twopi;
    return (double)p;
}

int cb_mixer_create(double dphase, double phase, cb_mixer **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(std::isfinite(dphase) && std::isfinite(phase), CB_ERR_INVALID_ARG, "mixer: non-finite phase");
    int rc = ensure_device();
    if (rc) return rc;
    cb_mixer *h = new (std::nothrow) cb_mixer();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->phase = phase;
    h->dphase = wrap_dphase(dphase);
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete h;
        return cuda_fail(e, "cudaStreamCreateWithFlags", __FILE__, __LINE__);
    }
    if (h->pipe.init(h->stream)) {
        cudaStreamDestroy(h->stream);
        delete h;
        return CB_ERR_CUDA;
    }
    *out = h;
    return CB_OK;
}

int cb_mixer_destroy(cb_mixer *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    h->pipe.destroy();
    cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_mixer_run_dev(cb_mixer *h, const float *d_in, size_t n, float *d_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    int rc = launch_mixer(reinterpret_cast<const float2 *>(d_in), reinterpret_cast<float2 *>(d_out), n, h->phase,
                          h->dphase, pick_stream(stream, h->stream));
    if (rc) return rc;
    h->phase = advance_phase(h->phase, h->dphase, n);
    return CB_OK;
}

int cb_mixer_run(cb_mixer *h, const float *in, size_t n, float *out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (n == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    const size_t chunk = n < HOST_CHUNK ? n : HOST_CHUNK;
    int rc = h->pipe.reserve(chunk * sizeof(float2), chunk * sizeof(float2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n * sizeof(float2), chunk * sizeof(float2), out, n * sizeof(float2), chunk * sizeof(float2));
    if (rc) return rc;
    const float2 *hin = reinterpret_cast<const float2 *>(in);
    float2 *hout = reinterpret_cast<float2 *>(out);
    size_t done = 0;
    for (int i = 0; done < n; ++i) {
        const int l = i & 1;
        const size_t m = n - done < chunk ? n - done : chunk;
        cudaStream_t s = h->pipe.lane[l];
        float2 *di = reinterpret_cast<float2 *>(h->pipe.in[l]), *dout = reinterpret_cast<float2 *>(h->pipe.out[l]);
        rc = h->pipe.h2d(l, di, hin + done, m * sizeof(float2));
        if (rc) return rc;
        rc = launch_mixer(di, dout, m, h->phase, h->dphase, s);
        if (rc) return rc;
        h->phase = advance_phase(h->phase, h->dphase, m);
        rc = h->pipe.d2h(l, hout + done, dout, m * sizeof(float2));
        if (rc) return rc;
        done += m;
    }
    return h->pipe.sync();
}

int cb_mixer_get_phase(const cb_mixer *h, double *phase, double *dphase)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (phase) *phase = h->phase;
    if (dphase) *dphase = h->dphase;
    return CB_OK;
}

int cb_mixer_set_phase(cb_mixer *h, double phase)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(std::isfinite(phase), CB_ERR_INVALID_ARG, "mixer: non-finite phase");
    h->phase = phase;
    return CB_OK;
}

// ============================================================================ FFT
static int upload_twiddles(size_t n, int inverse, float2 **dev)
{
    std::vector<float2> t(n);
    const long double sgn = inverse ? 2.0L : -2.0L;
    for (size_t k = 0; k < n; ++k) {
        const long double a = sgn * 3.14159265358979323846264338327950288L * (long double)k / (long double)n;
        t[k] = make_float2((float)cosl(a), (float)sinl(a));
    }
    CB_CUDA(cudaMalloc(dev, n * sizeof(float2)));
    CB_CUDA(cudaMemcpy(*dev, t.data(), n * sizeof(float2), cudaMemcpyHostToDevice));
    return CB_OK;
}

static int upload_fft2_table(int log2n, int inverse, float2 **dev)
{
    std::vector<float2> t(fft2_table_len(log2n));
    fft2_fill_table(log2n, inverse, t.data());
    CB_CUDA(cudaMalloc(dev, t.size() * sizeof(float2)));
    CB_CUDA(cudaMemcpy(*dev, t.data(), t.size() * sizeof(float2), cudaMemcpyHostToDevice));
    return CB_OK;
}

// in-place radix-2 transform in f64 (forward), for the one-off spectrum of the Bluestein chirp
static void host_fft_f64(std::vector<double> &re, std::vector<double> &im)
{
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) {
            std::swap(re[i], re[j]);
            std::swap(im[i], im[j]);
        }
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        const size_t half = len >> 1;
        std::vector<double> wr(half), wi(half);
        for (size_t k = 0; k < half; ++k) {
            const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)k / (long double)len;
            wr[k] = (double)cosl(a);
            wi[k] = (double)sinl(a);
        }
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < half; ++k) {
                const double xr = re[i + k + half] * wr[k] - im[i + k + half] * wi[k];
                const double xi = re[i + k + half] * wi[k] + im[i + k + half] * wr[k];
                re[i + k + half] = re[i + k] - xr;
                im[i + k + half] = im[i + k] - xi;
                re[i + k] += xr;
                im[i + k] += xi;
            }
    }
}

static int bluestein_setup(cb_fft *h, size_t n, int inverse)
{
    size_t m = 256;
    while (m < 2 * n - 1) m <<= 1;
    h->bl_m = m;
    // w[i] = e^{-/+ j pi i^2 / n}: i^2 reduced mod 2n in integers so that the angle stays exact for large i
    std::vector<float2> w(n);
    std::vector<double> br(m, 0.0), bi(m, 0.0);
    const long double sgn = inverse ? 1.0L : -1.0L;
    for (size_t i = 0; i < n; ++i) {
        const unsigned long long q = ((unsigned long long)i * i) % (2ull * n);
        const long double a = sgn * 3.14159265358979323846264338327950288L * (long double)q / (long double)n;
        const long double c = cosl(a), sn = sinl(a);
        w[i] = make_float2((float)c, (float)sn);
        br[i] = (double)c;
        bi[i] = (double)-sn;  // conj(w[i]) at +i and -i (wrapped)
        if (i) {
            br[m - i] = br[i];
            bi[m - i] = bi[i];
        }
    }
    host_fft_f64(br, bi);
    std::vector<float2> bs(m);
    for (size_t i = 0; i < m; ++i) bs[i] = make_float2((float)br[i], (float)bi[i]);
    CB_CUDA(cudaMalloc(&h->chirp, n * sizeof(float2)));
    CB_CUDA(cudaMemcpy(h->chirp, w.data(), n * sizeof(float2), cudaMemcpyHostToDevice));
    CB_CUDA(cudaMalloc(&h->bspec, m * sizeof(float2)));
    CB_CUDA(cudaMemcpy(h->bspec, bs.data(), m * sizeof(float2), cudaMemcpyHostToDevice));
    // work buffers: up to 16384 points one L2-sized buffer of spectra (the fused two-kernel form); beyond, the five-launch
    // form around the two-step transforms wants long batches (their persistent kernels ramp up and down per launch)
    h->bl_frames = ((size_t)(m <= 16384 ? 32 : 256) << 20) / (m * sizeof(float2));
    if (h->bl_frames < 1) h->bl_frames = 1;
    CB_CUDA(cudaMalloc(&h->bufa, h->bl_frames * m * sizeof(float2)));
    CB_CUDA(cudaMalloc(&h->bufb, h->bl_frames * m * sizeof(float2)));
    int rc = cb_fft_create(m, 0, &h->sub_f);
    if (rc) return rc;
    return cb_fft_create(m, 1, &h->sub_i);
}

int cb_fft_create(size_t fft_size, int inverse, cb_fft **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(fft_size >= 1, CB_ERR_INVALID_ARG, "fft: size must be >= 1");
    int rc = ensure_device();
    if (rc) return rc;
    const bool pow2 = (fft_size & (fft_size - 1)) == 0;
    int log2n = 0;
    while (((size_t)1 << log2n) < fft_size) ++log2n;
    int kind;
    int l1 = 0, l2 = 0;
    if (pow2 && log2n >= 3 && log2n <= 14) kind = FFT_SINGLE;  // one CTA per frame up to 16384 points (139 KiB of shared memory)
    else if (pow2 && log2n >= 15) {
        rc = fft_plan_split(fft_size, &l1, &l2);
        CB_REQUIRE(rc == CB_OK, CB_ERR_UNSUPPORTED, "fft: size %zu > 2^20 is not provided", fft_size);
        kind = FFT_FOURSTEP;
    } else {
        // any other size (rustfft plans every length): O(N^2) with an exact table while that is cheap, else chirp-z
        const char *path = getenv("COMMS_B200_FFT_PATH");
        const bool force_direct = path && strcmp(path, "direct") == 0 && fft_size <= 4096;
        CB_REQUIRE(fft_size <= ((size_t)1 << 19), CB_ERR_UNSUPPORTED,
                   "fft: non power-of-two size %zu > 2^19 is not provided", fft_size);
        kind = (fft_size <= 128 || force_direct) ? FFT_DIRECT : FFT_BLUESTEIN;
    }
    cb_fft *h = new (std::nothrow) cb_fft();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->tw = h->tw1 = h->tw2 = h->tw16 = h->tw16a = h->tw16b = h->scratch = nullptr;
    h->sub_f = h->sub_i = nullptr;
    h->chirp = h->bspec = h->bufa = h->bufb = nullptr;
    h->bl_m = h->bl_frames = 0;
    h->stream = nullptr;
    h->plan = FftPlanDev{};
    h->plan.kind = kind;
    h->plan.inverse = inverse ? 1 : 0;
    h->plan.n = fft_size;
    h->plan.log2n = log2n;
    h->plan.log2n1 = l1;
    h->plan.log2n2 = l2;
#define FFT_TRY(expr)                 \
    do {                              \
        int rc__ = (expr);            \
        if (rc__) {                   \
            cb_fft_destroy(h);        \
            return rc__;              \
        }                             \
    } while (0)
    {
        cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            h->stream = nullptr;
            cb_fft_destroy(h);
            return cuda_fail(e, "cudaStreamCreateWithFlags", __FILE__, __LINE__);
        }
    }
    FFT_TRY(h->pipe.init(h->stream));
    if (kind == FFT_BLUESTEIN) {
        FFT_TRY(bluestein_setup(h, fft_size, inverse));
        *out = h;
        return CB_OK;
    }
    FFT_TRY(upload_twiddles(fft_size, inverse, &h->tw));
    if (kind == FFT_SINGLE && log2n >= 4) FFT_TRY(upload_fft2_table(log2n, inverse, &h->tw16));
    if (kind == FFT_FOURSTEP) {
        FFT_TRY(upload_twiddles((size_t)1 << l1, inverse, &h->tw1));
        FFT_TRY(upload_twiddles((size_t)1 << l2, inverse, &h->tw2));
        // the fused two-step kernels keep the intermediate in a ring of scratch frames that stays in L2
        // (48 MiB measured best at every size, each CTA holding two tickets: profiles/r03h_fft65536_variants.txt; that is
        // 192 / 96 / 48 / 24 / 12 / 6 frames of 2^15 .. 2^20 points); the four-step fallback uses the same buffer in groups
        // of frames
        size_t scratch_mb = 48;
        FFT_TRY(upload_fft2_table(l1, inverse, &h->tw16a));
        FFT_TRY(upload_fft2_table(l2, inverse, &h->tw16b));
        h->plan.big = 1;
        if (const char *e = getenv("COMMS_B200_FFT_PATH"))
            if (strcmp(e, "fourstep") == 0) h->plan.big = 0;
        if (const char *e = getenv("COMMS_B200_FFT_SCRATCH_MB")) scratch_mb = (size_t)atol(e) > 0 ? (size_t)atol(e) : scratch_mb;
        size_t frames = (scratch_mb << 20) / (fft_size * sizeof(float2));
        if (frames < 1) frames = 1;
        if (fft_size == 65536) FFT_TRY(upload_fft2_table(12, inverse, &h->tw16));  // rows of the 16 x 4096 two-pass form
        h->plan.scratch_frames = frames;
        cudaError_t e = cudaMalloc(&h->scratch, frames * fft_size * sizeof(float2));
        if (e != cudaSuccess) {
            cb_fft_destroy(h);
            return cuda_fail(e, "cudaMalloc(scratch)", __FILE__, __LINE__);
        }
    }
#undef FFT_TRY
    h->plan.tw = h->tw;
    h->plan.tw1 = h->tw1;
    h->plan.tw2 = h->tw2;
    h->plan.tw16 = h->tw16;
    h->plan.tw16a = h->tw16a;
    h->plan.tw16b = h->tw16b;
    h->plan.scratch = h->scratch;
    // 65536 points.  COMMS_B200_FFT_PATH = rows (default: one persistent kernel over a 256 x 256 split, intermediate in
    // an L2-resident ring, K5-R) | rows2 (same two steps as two launches with a batch-sized scratch) | cluster (one HBM
    // pass on 8-CTA clusters, K5-C; also the fallback when an allocation fails) | cluster1 / cluster2 (its other
    // exchange synchronisations) | cluster16 | twopass | fourstep | cpipe | rowspf (K5-R2: rows with TMA-prefetched items)
    if (fft_size == 65536) {
        const char *path = getenv("COMMS_B200_FFT_PATH");
        h->plan.cluster_tpt = 6;
        if (path && strcmp(path, "cluster") == 0) h->plan.cluster_tpt = 3;
        if (path && strcmp(path, "cluster2") == 0) h->plan.cluster_tpt = 2;
        if (path && strcmp(path, "cluster16") == 0) h->plan.cluster_tpt = 4;  // 16-CTA clusters, 4 CTAs per SM
        if (path && strcmp(path, "twopass") == 0) h->plan.cluster_tpt = 5;    // 16 x 4096, two streaming passes
        if (path && strcmp(path, "rows") == 0) h->plan.cluster_tpt = 6;       // 256 x 256, fused persistent kernel, L2 ring
        if (path && strcmp(path, "rows2") == 0) h->plan.cluster_tpt = 7;      // 256 x 256, two launches, batch-sized scratch
        if (path && strcmp(path, "big") == 0) h->plan.cluster_tpt = 8;        // the generic fused two-step kernel (K5-B)
        if (path && strcmp(path, "cpipe") == 0) h->plan.cluster_tpt = 9;      // persistent pipelined 8-CTA clusters (K5-P)
        if (path && strcmp(path, "rowspf") == 0) h->plan.cluster_tpt = 10;    // rows with the next item's points prefetched (K5-R2)
    }
    *out = h;
    return CB_OK;
}

int cb_fft_destroy(cb_fft *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    if (h->tw) cudaFree(h->tw);
    if (h->tw1) cudaFree(h->tw1);
    if (h->tw2) cudaFree(h->tw2);
    if (h->tw16) cudaFree(h->tw16);
    if (h->sub_f) cb_fft_destroy(h->sub_f);
    if (h->sub_i) cb_fft_destroy(h->sub_i);
    if (h->chirp) cudaFree(h->chirp);
    if (h->bspec) cudaFree(h->bspec);
    if (h->bufa) cudaFree(h->bufa);
    if (h->bufb) cudaFree(h->bufb);
    if (h->tw16a) cudaFree(h->tw16a);
    if (h->tw16b) cudaFree(h->tw16b);
    if (h->scratch) cudaFree(h->scratch);
    if (h->plan.flags) cudaFree(h->plan.flags);

    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_fft_size(const cb_fft *h, size_t *fft_size, int *inverse)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (fft_size) *fft_size = h->plan.n;
    if (inverse) *inverse = h->plan.inverse;
    return CB_OK;
}

// 65536-point "rows" paths.  Fused (mode 6): the scratch is a fixed L2-sized ring allocated with the plan; only the
// per-frame dependency counters grow with the batch.  Two-launch (mode 7): the scratch is as large as the batch.
// Both grow on demand (cudaFree waits for work that may still use the old buffer); when an allocation fails the
// handle switches to the one-pass cluster kernel, which needs neither.
static void fft_prepare_scratch(cb_fft *h, size_t nframes)
{
    if (h->plan.kind != FFT_FOURSTEP) return;
    const bool big = h->plan.big && (h->plan.n != 65536 || h->plan.cluster_tpt == 8);
    if ((big || (h->plan.n == 65536 && (h->plan.cluster_tpt == 6 || h->plan.cluster_tpt == 10))) && h->plan.flags_frames < nframes) {
        if (h->plan.flags) cudaFree(h->plan.flags);
        h->plan.flags = nullptr;
        h->plan.flags_frames = 0;
        if (cudaMalloc(&h->plan.flags, (4 + 2 * nframes) * sizeof(unsigned)) != cudaSuccess) {
            cudaGetLastError();
            h->plan.flags = nullptr;
            h->plan.big = 0;  // four-step
            if (h->plan.n == 65536) h->plan.cluster_tpt = 3;
            return;
        }
        h->plan.flags_frames = nframes;
    }
    if (h->plan.n == 65536 && h->plan.cluster_tpt == 7 && h->plan.scratch_frames < nframes) {
        if (h->scratch) cudaFree(h->scratch);
        h->scratch = nullptr;
        h->plan.scratch = nullptr;
        h->plan.scratch_frames = 0;
        if (cudaMalloc(&h->scratch, nframes * h->plan.n * sizeof(float2)) != cudaSuccess) {
            cudaGetLastError();
            h->scratch = nullptr;
            h->plan.cluster_tpt = 3;
            return;
        }
        h->plan.scratch = h->scratch;
        h->plan.scratch_frames = nframes;
    }
}

// one batch of frames on stream s, whatever the plan kind
static int fft_exec(cb_fft *h, const float2 *in, float2 *out, size_t nframes, cudaStream_t s)
{
    if (h->plan.kind != FFT_BLUESTEIN) {
        fft_prepare_scratch(h, nframes);
        return launch_fft(h->plan, in, out, nframes, s);
    }
    const uint32_t N = (uint32_t)h->plan.n, M = (uint32_t)h->bl_m;
    // COMMS_B200_FFT_CHIRPZ=split: the five-launch form (element-wise kernels around the sub-plans) for every size
    static const bool bl_split = [] { const char *e = getenv("COMMS_B200_FFT_CHIRPZ"); return e && strcmp(e, "split") == 0; }();
    for (size_t done = 0; done < nframes;) {
        const size_t g = nframes - done < h->bl_frames ? nframes - done : h->bl_frames;
        if (M <= 16384 && h->sub_f->tw16 && h->sub_i->tw16 && !bl_split) {  // two kernels per group, spectra in bufa
            int rc = launch_bluestein_fused(in + done * N, h->chirp, h->bspec, h->bufa, out + done * N, N, h->sub_f->plan.log2n,
                                            h->sub_f->tw16, h->sub_i->tw16, g, s);
            if (rc) return rc;
            done += g;
            continue;
        }
        int rc = launch_bluestein_pre(in + done * N, h->chirp, h->bufa, N, M, g, s);
        if (!rc) rc = fft_exec(h->sub_f, h->bufa, h->bufb, g, s);
        if (!rc) rc = launch_bluestein_mul(h->bufb, h->bspec, M, g, s);
        if (!rc) rc = fft_exec(h->sub_i, h->bufb, h->bufa, g, s);
        if (!rc) rc = launch_bluestein_post(h->bufa, h->chirp, out + done * N, N, M, g, s);
        if (rc) return rc;
        done += g;
    }
    return CB_OK;
}

int cb_fft_run_dev(cb_fft *h, const float *d_in, size_t n_in, float *d_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    // rustfft asserts input.len() == fft_size (src/fft/mod.rs:86): a wrong length is an error
    CB_REQUIRE(n_in > 0 && n_in % h->plan.n == 0, CB_ERR_SIZE, "fft: input length %zu is not a multiple of fft_size %zu",
               n_in, h->plan.n);
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_NO_ALIAS(d_in, n_in * sizeof(float2), d_out, n_in * sizeof(float2), "fft");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    // the scratch ring, its counters and the chirp-z work buffers are per handle: order calls across streams
    const bool shared = h->plan.kind == FFT_FOURSTEP || h->plan.kind == FFT_BLUESTEIN;
    int rc = shared ? h->last.begin(s) : CB_OK;
    if (rc) return rc;
    rc = fft_exec(h, reinterpret_cast<const float2 *>(d_in), reinterpret_cast<float2 *>(d_out), n_in / h->plan.n, s);
    if (rc) return rc;
    return shared ? h->last.end(s) : CB_OK;
}

int cb_fft_run(cb_fft *h, const float *in, size_t n_in, float *out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(n_in > 0 && n_in % h->plan.n == 0, CB_ERR_SIZE, "fft: input length %zu is not a multiple of fft_size %zu",
               n_in, h->plan.n);
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    const size_t N = h->plan.n;
    size_t chunk = HOST_CHUNK / N * N;
    if (chunk == 0) chunk = N;
    if (n_in < chunk) chunk = n_in;
    int rc = h->last.sync();
    if (rc) return rc;
    rc = h->pipe.reserve(chunk * sizeof(float2), chunk * sizeof(float2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n_in * sizeof(float2), chunk * sizeof(float2), out, n_in * sizeof(float2), chunk * sizeof(float2));
    if (rc) return rc;
    const float2 *hin = reinterpret_cast<const float2 *>(in);
    float2 *hout = reinterpret_cast<float2 *>(out);
    size_t done = 0;
    for (int i = 0; done < n_in; ++i) {
        const int l = i & 1;
        const size_t m = n_in - done < chunk ? n_in - done : chunk;
        cudaStream_t s = h->pipe.lane[l];
        float2 *di = reinterpret_cast<float2 *>(h->pipe.in[l]), *dout = reinterpret_cast<float2 *>(h->pipe.out[l]);
        rc = h->pipe.h2d(l, di, hin + done, m * sizeof(float2));
        if (rc) return rc;
        if ((h->plan.kind == FFT_FOURSTEP || h->plan.kind == FFT_BLUESTEIN) && i > 0) {
            // the scratch / work buffers are shared by both lanes: serialise the kernels
            CB_CUDA(cudaStreamSynchronize(h->pipe.lane[l ^ 1]));
        }
        rc = fft_exec(h, di, dout, m / N, s);
        if (rc) return rc;
        rc = h->pipe.d2h(l, hout + done, dout, m * sizeof(float2));
        if (rc) return rc;
        done += m;
    }
    return h->pipe.sync();
}

// i16 IQ frames in (IQBatchInput, src/io/raw_iq.rs:78-140), f32 spectra out: x = in_scale * (i16 as f32)
// i16 IQ in: the transforms that read the samples themselves (single-kernel sizes, 65536 points) widen them in their
// first loads; the others get a widening pass into the lane's scratch first
static int fft_exec_iq16(cb_fft *h, const int16_t *d_in, float in_scale, float2 *d_out, size_t nframes, int lane, cudaStream_t s)
{
    if (h->plan.kind != FFT_BLUESTEIN) {
        fft_prepare_scratch(h, nframes);
        if (fft_fuses_iq16(h->plan, nframes)) return launch_fft_iq16(h->plan, d_in, in_scale, d_out, nframes, s);
    }
    const size_t n = nframes * h->plan.n;
    int rc = h->pipe.reserve_aux(n * sizeof(float2), 0);
    if (rc) return rc;
    float2 *wide = reinterpret_cast<float2 *>(h->pipe.aux_in[lane]);
    rc = launch_convert_i16(d_in, reinterpret_cast<float *>(wide), 2 * n, in_scale, s);
    if (rc) return rc;
    return fft_exec(h, wide, d_out, nframes, s);
}

int cb_fft_run_dev_iq16(cb_fft *h, const int16_t *d_in, size_t n_in, float in_scale, float *d_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(n_in > 0 && n_in % h->plan.n == 0, CB_ERR_SIZE, "fft: input length %zu is not a multiple of fft_size %zu",
               n_in, h->plan.n);
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_NO_ALIAS(d_in, n_in * 2 * sizeof(int16_t), d_out, n_in * sizeof(float2), "fft");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);  // the widened-input scratch is per handle
    if (rc) return rc;
    rc = fft_exec_iq16(h, d_in, in_scale, reinterpret_cast<float2 *>(d_out), n_in / h->plan.n, 0, s);
    if (rc) return rc;
    return h->last.end(s);
}

int cb_fft_run_iq16(cb_fft *h, const int16_t *in, size_t n_in, float in_scale, float *out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(n_in > 0 && n_in % h->plan.n == 0, CB_ERR_SIZE, "fft: input length %zu is not a multiple of fft_size %zu",
               n_in, h->plan.n);
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    const size_t N = h->plan.n, IQ = 2 * sizeof(int16_t);
    size_t chunk = HOST_CHUNK / N * N;
    if (chunk == 0) chunk = N;
    if (n_in < chunk) chunk = n_in;
    int rc = h->last.sync();
    if (rc) return rc;
    rc = h->pipe.reserve(chunk * IQ, chunk * sizeof(float2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n_in * IQ, chunk * IQ, out, n_in * sizeof(float2), chunk * sizeof(float2));
    if (rc) return rc;
    const char *hin = reinterpret_cast<const char *>(in);
    float2 *hout = reinterpret_cast<float2 *>(out);
    size_t done = 0;
    for (int i = 0; done < n_in; ++i) {
        const int l = i & 1;
        const size_t m = n_in - done < chunk ? n_in - done : chunk;
        cudaStream_t s = h->pipe.lane[l];
        float2 *dout = reinterpret_cast<float2 *>(h->pipe.out[l]);
        rc = h->pipe.h2d(l, h->pipe.in[l], hin + done * IQ, m * IQ);
        if (rc) return rc;
        if ((h->plan.kind == FFT_FOURSTEP || h->plan.kind == FFT_BLUESTEIN) && i > 0) CB_CUDA(cudaStreamSynchronize(h->pipe.lane[l ^ 1]));
        rc = fft_exec_iq16(h, reinterpret_cast<const int16_t *>(h->pipe.in[l]), in_scale, dout, m / N, l, s);
        if (rc) return rc;
        rc = h->pipe.d2h(l, hout + done, dout, m * sizeof(float2));
        if (rc) return rc;
        done += m;
    }
    return h->pipe.sync();
}

// ============================================================================ FFT over Complex<f64>
// The plan picks its path from the size alone (fft64_core.cuh, "plan shape"); every rounding is in the host/device
// functions of fft64_core.cuh, so the CPU emulation reproduces the bits.
enum { F64_DIRECT = 0, F64_FRAMES = 1, F64_TWOSTEP = 2, F64_CHIRPZ = 3 };

struct cb_fft_f64 {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    size_t n;
    int inverse;
    int kind;
    unsigned log2n;               // powers of two: log2 n; chirp-z: log2 m
    size_t m;                     // chirp-z: the padded power of two
    double2 *tw;                  // n-entry twiddle table of the plan's sign (chirp-z: m entries, forward)
    double2 *tw_inv;              // chirp-z: m entries, inverse
    double2 *chirp, *bspec;       // chirp-z: n chirp values, m spectrum values (1/m folded in)
    double2 *scratch, *bufa, *bufb;  // two-step intermediate / chirp-z work buffers, `group` frames each
    size_t group;
    LastUse last;
};

static int f64_upload(const std::vector<f64fft::z64> &v, double2 **dev)
{
    CB_CUDA(cudaMalloc(dev, v.size() * sizeof(double2)));
    CB_CUDA(cudaMemcpy(*dev, v.data(), v.size() * sizeof(double2), cudaMemcpyHostToDevice));
    return CB_OK;
}

// Transforms of 2^L points (L >= 3): one frame-kernel launch up to 2^FRAME_MAX_LOG2, else two launches per group of
// frames through the scratch: N1-point transforms down the columns (stride N2) with the inter-step twiddle tw[k1 n2]
// applied on the way out, then N2-point transforms of the rows, stored transposed (X[k1 + N1 k2]).
static int f64_pow2(unsigned L, const double2 *tw, int inverse, const double2 *in, double2 *out, size_t frames,
                    double2 *scratch, size_t group, cudaStream_t s)
{
    const size_t N = (size_t)1 << L;
    if (L <= f64fft::FRAME_MAX_LOG2) {
        const Fft64Cols a{in, out, tw, nullptr, 1, N, 0, 1, N, 0, 1, L, (unsigned)frames, 1};
        return launch_fft64_cols(a, inverse, s);
    }
    const unsigned L1 = L / 2, L2 = L - L1;
    const size_t N1 = (size_t)1 << L1, N2 = (size_t)1 << L2;
    for (size_t done = 0; done < frames;) {
        const size_t g = frames - done < group ? frames - done : group;
        const Fft64Cols a{in + done * N, scratch, tw, tw, N2, 1, N, 1, N1, N, (unsigned)N2, L1, (unsigned)N2, g};
        int rc = launch_fft64_cols(a, inverse, s);
        if (rc) return rc;
        const Fft64Cols b{scratch, out + done * N, tw, nullptr, N1, 1, N, N1, 1, N, (unsigned)N1, L2, (unsigned)N1, g};
        rc = launch_fft64_cols(b, inverse, s);
        if (rc) return rc;
        done += g;
    }
    return CB_OK;
}

static int f64_exec(cb_fft_f64 *h, const double2 *in, double2 *out, size_t frames, cudaStream_t s)
{
    const unsigned N = (unsigned)h->n;
    if (h->kind == F64_DIRECT) return launch_fft64_direct(in, out, h->tw, N, frames, s);
    if (h->kind != F64_CHIRPZ) return f64_pow2(h->log2n, h->tw, h->inverse, in, out, frames, h->scratch, h->group, s);
    const unsigned M = (unsigned)h->m;
    for (size_t done = 0; done < frames;) {
        const size_t g = frames - done < h->group ? frames - done : h->group;
        int rc = launch_fft64_chirp_pre(in + done * N, h->chirp, h->bufa, N, M, g, s);
        if (!rc) rc = f64_pow2(h->log2n, h->tw, 0, h->bufa, h->bufb, g, h->scratch, g, s);
        if (!rc) rc = launch_fft64_chirp_mul(h->bufb, h->bspec, M, g, s);
        if (!rc) rc = f64_pow2(h->log2n, h->tw_inv, 1, h->bufb, h->bufa, g, h->scratch, g, s);
        if (!rc) rc = launch_fft64_chirp_post(h->bufa, h->chirp, out + done * N, N, M, g, s);
        if (rc) return rc;
        done += g;
    }
    return CB_OK;
}

int cb_fft_f64_create(size_t fft_size, int inverse, cb_fft_f64 **out)
{
    using namespace f64fft;
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(fft_size >= 1, CB_ERR_INVALID_ARG, "fft_f64: size must be >= 1");
    const bool pow2 = (fft_size & (fft_size - 1)) == 0;
    CB_REQUIRE(fft_size <= ((size_t)1 << (pow2 ? 20 : 19)), CB_ERR_UNSUPPORTED, "fft_f64: size %zu is not provided",
               fft_size);
    int rc = ensure_device();
    if (rc) return rc;
    cb_fft_f64 *h = new (std::nothrow) cb_fft_f64();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->n = fft_size;
    h->inverse = inverse ? 1 : 0;
    unsigned L = 0;
    while (((size_t)1 << L) < fft_size) ++L;
    h->log2n = L;
    if (pow2 && L >= 3) h->kind = L <= FRAME_MAX_LOG2 ? F64_FRAMES : F64_TWOSTEP;
    else if (pow2 || fft_size <= DIRECT_MAX) h->kind = F64_DIRECT;
    else {
        h->kind = F64_CHIRPZ;
        h->m = 8;
        while (h->m < 2 * fft_size - 1) h->m <<= 1;
        h->log2n = 0;
        while (((size_t)1 << h->log2n) < h->m) ++h->log2n;
    }
    // two-step and chirp-z work in groups of frames whose buffers take 64 MiB each
    const size_t span = h->kind == F64_CHIRPZ ? h->m : fft_size;
    h->group = ((size_t)64 << 20) / (span * sizeof(double2));
    if (h->group < 1) h->group = 1;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        h->stream = nullptr;
        cb_fft_f64_destroy(h);
        return cuda_fail(e, "cudaStreamCreateWithFlags", __FILE__, __LINE__);
    }
    rc = h->pipe.init(h->stream);
    if (!rc && h->kind != F64_CHIRPZ) rc = f64_upload(twiddle_table(fft_size, h->inverse), &h->tw);
    if (!rc && h->kind == F64_CHIRPZ) {
        std::vector<z64> chirp, bspec;
        chirp_tables(fft_size, h->m, h->inverse, chirp, bspec);
        rc = f64_upload(chirp, &h->chirp);
        if (!rc) rc = f64_upload(bspec, &h->bspec);
        if (!rc) rc = f64_upload(twiddle_table(h->m, 0), &h->tw);
        if (!rc) rc = f64_upload(twiddle_table(h->m, 1), &h->tw_inv);
        if (!rc && cudaMalloc(&h->bufa, h->group * h->m * sizeof(double2)) != cudaSuccess) rc = CB_ERR_OOM;
        if (!rc && cudaMalloc(&h->bufb, h->group * h->m * sizeof(double2)) != cudaSuccess) rc = CB_ERR_OOM;
    }
    if (!rc && h->log2n > FRAME_MAX_LOG2 && cudaMalloc(&h->scratch, h->group * span * sizeof(double2)) != cudaSuccess)
        rc = CB_ERR_OOM;
    if (rc) {
        if (rc == CB_ERR_OOM) {
            cudaGetLastError();
            set_error("fft_f64: work buffer allocation failed");
        }
        cb_fft_f64_destroy(h);
        return rc;
    }
    *out = h;
    return CB_OK;
}

int cb_fft_f64_destroy(cb_fft_f64 *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    for (double2 *p : {h->tw, h->tw_inv, h->chirp, h->bspec, h->scratch, h->bufa, h->bufb})
        if (p) cudaFree(p);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_fft_f64_size(const cb_fft_f64 *h, size_t *fft_size, int *inverse)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (fft_size) *fft_size = h->n;
    if (inverse) *inverse = h->inverse;
    return CB_OK;
}

int cb_fft_f64_run_dev(cb_fft_f64 *h, const double *d_in, size_t n_in, double *d_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(n_in > 0 && n_in % h->n == 0, CB_ERR_SIZE, "fft_f64: input length %zu is not a multiple of fft_size %zu",
               n_in, h->n);
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(((reinterpret_cast<uintptr_t>(d_in) | reinterpret_cast<uintptr_t>(d_out)) & 15) == 0, CB_ERR_INVALID_ARG,
               "fft_f64: d_in and d_out must be 16-byte aligned");  // read and written as double2
    CB_NO_ALIAS(d_in, n_in * sizeof(double2), d_out, n_in * sizeof(double2), "fft_f64");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);  // the two-step scratch and the chirp-z work buffers are per handle
    if (rc) return rc;
    rc = f64_exec(h, reinterpret_cast<const double2 *>(d_in), reinterpret_cast<double2 *>(d_out), n_in / h->n, s);
    if (rc) return rc;
    return h->last.end(s);
}

int cb_fft_f64_run(cb_fft_f64 *h, const double *in, size_t n_in, double *out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(n_in > 0 && n_in % h->n == 0, CB_ERR_SIZE, "fft_f64: input length %zu is not a multiple of fft_size %zu",
               n_in, h->n);
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    const size_t N = h->n;
    size_t chunk = HOST_CHUNK / N * N;
    if (chunk == 0) chunk = N;
    if (n_in < chunk) chunk = n_in;
    int rc = h->last.sync();
    if (rc) return rc;
    rc = h->pipe.reserve(chunk * sizeof(double2), chunk * sizeof(double2));
    if (rc) return rc;
    rc = h->pipe.begin_call(in, n_in * sizeof(double2), chunk * sizeof(double2), out, n_in * sizeof(double2),
                            chunk * sizeof(double2));
    if (rc) return rc;
    const double2 *hin = reinterpret_cast<const double2 *>(in);
    double2 *hout = reinterpret_cast<double2 *>(out);
    const bool shared = h->kind == F64_TWOSTEP || h->kind == F64_CHIRPZ;
    size_t done = 0;
    for (int i = 0; done < n_in; ++i) {
        const int l = i & 1;
        const size_t m = n_in - done < chunk ? n_in - done : chunk;
        cudaStream_t s = h->pipe.lane[l];
        double2 *di = reinterpret_cast<double2 *>(h->pipe.in[l]), *dout = reinterpret_cast<double2 *>(h->pipe.out[l]);
        rc = h->pipe.h2d(l, di, hin + done, m * sizeof(double2));
        if (rc) return rc;
        if (shared && i > 0) CB_CUDA(cudaStreamSynchronize(h->pipe.lane[l ^ 1]));  // one scratch for both lanes
        rc = f64_exec(h, di, dout, m / N, s);
        if (rc) return rc;
        rc = h->pipe.d2h(l, hout + done, dout, m * sizeof(double2));
        if (rc) return rc;
        done += m;
    }
    return h->pipe.sync();
}

// ============================================================================ FM demod
int cb_fm_create(cb_fm **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    int rc = ensure_device();
    if (rc) return rc;
    cb_fm *h = new (std::nothrow) cb_fm();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->cur = 0;
    h->prev[0] = h->prev[1] = nullptr;
    h->stream = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&h->prev[0], sizeof(float2));
    if (e == cudaSuccess) e = cudaMalloc(&h->prev[1], sizeof(float2));
    if (e == cudaSuccess) e = cudaMemset(h->prev[0], 0, sizeof(float2));  // FM::default (analog.rs:43-47)
    if (e == cudaSuccess) e = cudaMemset(h->prev[1], 0, sizeof(float2));
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);  // the handle's non-blocking stream does not wait for it
    if (e != cudaSuccess || h->pipe.init(h->stream)) {
        cb_fm_destroy(h);
        return e != cudaSuccess ? cuda_fail(e, "fm create", __FILE__, __LINE__) : CB_ERR_CUDA;
    }
    *out = h;
    return CB_OK;
}

int cb_fm_destroy(cb_fm *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    for (int i = 0; i < 2; ++i)
        if (h->prev[i]) cudaFree(h->prev[i]);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_fm_run_dev(cb_fm *h, const float *d_in, size_t n, float *d_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_NO_ALIAS(d_in, n * sizeof(float2), d_out, n * sizeof(float), "fm");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);
    if (rc) return rc;
    rc = launch_fm(reinterpret_cast<const float2 *>(d_in), d_out, n, h->prev[h->cur], h->prev[h->cur ^ 1], s);
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

int cb_fm_run(cb_fm *h, const float *in, size_t n, float *out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (n == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    int rc = h->pipe.reserve(n * sizeof(float2), n * sizeof(float));
    if (rc) return rc;
    cudaStream_t s = h->pipe.lane[0];
    CB_CUDA(cudaMemcpyAsync(h->pipe.in[0], in, n * sizeof(float2), cudaMemcpyHostToDevice, s));
    rc = cb_fm_run_dev(h, reinterpret_cast<const float *>(h->pipe.in[0]), n, reinterpret_cast<float *>(h->pipe.out[0]), s);
    if (rc) return rc;
    CB_CUDA(cudaMemcpyAsync(out, h->pipe.out[0], n * sizeof(float), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
    return CB_OK;
}

// ============================================================================ fused bank
int cb_chain_create(size_t channels, const double *dphase, const double *phase, const float *taps, size_t ntaps,
                    uint32_t decim, int with_fm, cb_chain **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(channels >= 1 && channels <= 65535, CB_ERR_INVALID_ARG, "chain: channels must be 1..65535");
    CB_REQUIRE(taps && ntaps >= 1, CB_ERR_INVALID_ARG, "chain: taps required");
    int rc = ensure_device();
    if (rc) return rc;
    const float2 *t = reinterpret_cast<const float2 *>(taps);
    bool cplx = false;
    for (size_t k = 0; k < ntaps; ++k)
        if (t[k].y != 0.f) cplx = true;
    CB_REQUIRE(ntaps * (cplx ? 2 : 1) <= (size_t)CHAIN_MAX_TAP_SLOTS, CB_ERR_UNSUPPORTED,
               "chain: at most %d real or %d complex taps", CHAIN_MAX_TAP_SLOTS, CHAIN_MAX_TAP_SLOTS / 2);
    cb_chain *h = new (std::nothrow) cb_chain();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->channels = channels;
    h->mix = dphase != nullptr;
    h->fm = with_fm != 0;
    h->cplx = cplx;
    h->ntaps = (uint32_t)ntaps;
    h->decim = decim == 0 ? 1 : decim;
    // >= 128 samples of raw history per channel: the TMA-staged kernel bulk-copies whole halo chunks from it
    h->hist_len = (uint32_t)round_up(ntaps > 128 ? ntaps : 128, 2);
    h->cur = 0;
    memset(&h->taps, 0, sizeof h->taps);
    for (size_t k = 0; k < ntaps; ++k) {
        if (cplx) {
            h->taps.t[2 * k] = make_float2(t[k].x, t[k].x);
            h->taps.t[2 * k + 1] = make_float2(t[k].y, t[k].y);
        } else {
            h->taps.t[k] = make_float2(t[k].x, t[k].x);
        }
    }
    h->phase[0] = h->phase[1] = h->dphase = nullptr;
    h->hist[0] = h->hist[1] = h->prev[0] = h->prev[1] = nullptr;
    h->stream = nullptr;
    h->cscratch = nullptr;
    h->cscratch_len = 0;
    h->tc_img = nullptr;
    h->tc_seam = nullptr;
    h->tc_seam_len = 0;
    h->tc_inv_scale = 1.f;
    h->tc_dc = 0.f;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess && chain_tc_supported(h->ntaps, h->decim, h->mix, h->cplx)) {
        std::vector<unsigned char> img(chain_tc_image_bytes());
        std::vector<float> re(ntaps);
        for (size_t k = 0; k < ntaps; ++k) re[k] = t[k].x;
        chain_tc_build_image(re.data(), (uint32_t)ntaps, img.data(), &h->tc_inv_scale, &h->tc_dc);
        e = cudaMalloc(&h->tc_img, img.size());
        if (e == cudaSuccess) e = cudaMemcpy(h->tc_img, img.data(), img.size(), cudaMemcpyHostToDevice);
    }
    const size_t hb = channels * h->hist_len * sizeof(float2);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaMalloc(&h->hist[i], hb);
        if (e == cudaSuccess) e = cudaMemset(h->hist[i], 0, hb);
        if (e == cudaSuccess) e = cudaMalloc(&h->prev[i], channels * sizeof(float2));
        if (e == cudaSuccess) e = cudaMemset(h->prev[i], 0, channels * sizeof(float2));
        if (e == cudaSuccess) e = cudaMalloc(&h->phase[i], channels * sizeof(double));
        if (e == cudaSuccess) e = cudaMemset(h->phase[i], 0, channels * sizeof(double));
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);  // the memsets above: non-blocking streams do not wait for them
    if (e == cudaSuccess) e = cudaMalloc(&h->dphase, channels * sizeof(double));
    if (e == cudaSuccess && h->mix) {
        std::vector<double> d(channels), p(channels, 0.0);
        for (size_t c = 0; c < channels; ++c) {
            d[c] = wrap_dphase(dphase[c]);
            if (phase) p[c] = phase[c];
        }
        e = cudaMemcpy(h->dphase, d.data(), channels * sizeof(double), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(h->phase[0], p.data(), channels * sizeof(double), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess || h->pipe.init(h->stream)) {
        cb_chain_destroy(h);
        return e != cudaSuccess ? cuda_fail(e, "chain create", __FILE__, __LINE__) : CB_ERR_CUDA;
    }
    *out = h;
    return CB_OK;
}

int cb_chain_destroy(cb_chain *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    for (int i = 0; i < 2; ++i) {
        if (h->hist[i]) cudaFree(h->hist[i]);
        if (h->prev[i]) cudaFree(h->prev[i]);
        if (h->phase[i]) cudaFree(h->phase[i]);
    }
    if (h->dphase) cudaFree(h->dphase);
    if (h->cscratch) cudaFree(h->cscratch);
    if (h->tc_img) cudaFree(h->tc_img);
    if (h->tc_seam) cudaFree(h->tc_seam);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_chain_out_len(const cb_chain *h, size_t n_in, size_t *n_out)
{
    CB_REQUIRE(h && n_out, CB_ERR_INVALID_ARG, "NULL argument");
    *n_out = decim_len(n_in, h->decim);
    return CB_OK;
}

// d_in: complex-f32 input, or d_in8: (u8 I, u8 Q) byte pairs (exactly one of the two)
static int chain_run_dev_impl(cb_chain *h, const float *d_in, const uint8_t *d_in8, size_t n_in, float *d_out,
                              size_t out_cap, size_t *n_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = decim_len(n_in, h->decim);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE((d_in || d_in8) && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "chain: out_cap %zu < %zu outputs per channel", out_cap, no);
    CB_NO_ALIAS(d_in ? (const void *)d_in : (const void *)d_in8, h->channels * n_in * (d_in ? sizeof(float2) : 2), d_out,
                h->channels * no * (h->fm ? sizeof(float) : sizeof(float2)), "chain");
    CB_CUDA(cudaSetDevice(h->device));
    ChainArgs a;
    a.x = reinterpret_cast<const float2 *>(d_in);
    a.x8 = d_in8;
    a.out = d_out;
    a.phase_in = h->phase[h->cur];
    a.phase_out = h->phase[h->cur ^ 1];
    a.dphase = h->dphase;
    a.hist_in = h->hist[h->cur];
    a.hist_out = h->hist[h->cur ^ 1];
    a.prev_in = h->prev[h->cur];
    a.prev_out = h->prev[h->cur ^ 1];
    a.n_in = n_in;
    a.n_out = no;
    a.ntaps = h->ntaps;
    a.decim = h->decim;
    a.hist_len = h->hist_len;
    a.tc_img = h->tc_img;
    a.tc_inv_scale = h->tc_inv_scale;
    a.tc_dc = h->tc_dc;
    if (h->tc_img != nullptr && d_in8 != nullptr) {
        const size_t need = chain_tc_seam_entries(no, h->channels);
        if (h->tc_seam_len < need) {
            if (h->tc_seam) cudaFree(h->tc_seam);  // waits for launches that still use it
            h->tc_seam = nullptr;
            h->tc_seam_len = 0;
            if (cudaMalloc(&h->tc_seam, need * sizeof(float2)) == cudaSuccess) h->tc_seam_len = need;
            else (void)cudaGetLastError();  // without the scratch the CUDA-core kernel runs
        }
        a.tc_seam = h->tc_seam;
    }
    // outputs per CTA: keep the staged span around 48 KiB, whole multiples of 256 when possible
    size_t budget = (6144 > h->ntaps + h->decim ? 6144 - h->ntaps - h->decim : 0) / h->decim;
    size_t to = budget >= 256 ? budget / 256 * 256 : (budget ? budget : 1);
    if (to > 2048) to = 2048;
    if (to > no) to = no;
    a.tile_out = (unsigned)to;
    a.span_max = (unsigned)round_up((to + 1) * h->decim + h->ntaps, 2);
    CB_REQUIRE(ceil_div((size_t)a.span_max, (size_t)256) <= 64, CB_ERR_UNSUPPORTED,
               "chain: decimation %u with %u taps needs a span beyond the staged window", h->decim, h->ntaps);
    cudaStream_t s = pick_stream(stream, h->stream);
    {
        const int rcl = h->last.begin(s);
        if (rcl) return rcl;
    }
    if (d_in8 != nullptr && !chain_fuses_u8(a, h->cplx)) {  // no fused kernel for this shape: convert, then filter
        const size_t total = h->channels * n_in;
        if (h->cscratch_len < total) {
            if (h->cscratch) CB_CUDA(cudaFree(h->cscratch));
            h->cscratch = nullptr;
            h->cscratch_len = 0;
            CB_CUDA(cudaMalloc(&h->cscratch, total * sizeof(float2)));
            h->cscratch_len = total;
        }
        int rcc = launch_convert_u8(d_in8, reinterpret_cast<float *>(h->cscratch), 2 * total, s);
        if (rcc) return rcc;
        a.x = h->cscratch;
        a.x8 = nullptr;
    }
    int rc = launch_chain(a, h->taps, h->mix, h->fm, h->cplx, h->channels, s);
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

int cb_chain_run_dev(cb_chain *h, const float *d_in, size_t n_in, float *d_out, size_t out_cap, size_t *n_out,
                     void *stream)
{
    CB_REQUIRE(d_in || n_in == 0, CB_ERR_INVALID_ARG, "NULL data pointer");
    return chain_run_dev_impl(h, d_in, nullptr, n_in, d_out, out_cap, n_out, stream);
}

int cb_chain_run_u8_dev(cb_chain *h, const uint8_t *d_in, size_t n_in, float *d_out, size_t out_cap, size_t *n_out,
                        void *stream)
{
    CB_REQUIRE(d_in || n_in == 0, CB_ERR_INVALID_ARG, "NULL data pointer");
    return chain_run_dev_impl(h, nullptr, d_in, n_in, d_out, out_cap, n_out, stream);
}

int cb_chain_run_u8(cb_chain *h, const uint8_t *in, size_t n_in, float *out, size_t out_cap, size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = decim_len(n_in, h->decim);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "chain: out_cap %zu < %zu outputs per channel", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    const size_t in_bytes = h->channels * n_in * 2;
    const size_t out_bytes = h->channels * no * (h->fm ? sizeof(float) : sizeof(float2));
    int rc = h->pipe.reserve(in_bytes, out_bytes);
    if (rc) return rc;
    cudaStream_t s = h->pipe.lane[0];
    CB_CUDA(cudaMemcpyAsync(h->pipe.in[0], in, in_bytes, cudaMemcpyHostToDevice, s));
    rc = cb_chain_run_u8_dev(h, reinterpret_cast<const uint8_t *>(h->pipe.in[0]), n_in,
                             reinterpret_cast<float *>(h->pipe.out[0]), no, nullptr, s);
    if (rc) return rc;
    const size_t esz = h->fm ? sizeof(float) : sizeof(float2);
    CB_CUDA(cudaMemcpy2DAsync(out, out_cap * esz, h->pipe.out[0], no * esz, no * esz, h->channels, cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
    return CB_OK;
}

int cb_chain_run(cb_chain *h, const float *in, size_t n_in, float *out, size_t out_cap, size_t *n_out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    const size_t no = decim_len(n_in, h->decim);
    if (n_out) *n_out = no;
    if (n_in == 0) return CB_OK;
    CB_REQUIRE(in && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(out_cap >= no, CB_ERR_SIZE, "chain: out_cap %zu < %zu outputs per channel", out_cap, no);
    CB_CUDA(cudaSetDevice(h->device));
    const size_t in_bytes = h->channels * n_in * sizeof(float2);
    const size_t out_bytes = h->channels * no * (h->fm ? sizeof(float) : sizeof(float2));
    int rc = h->pipe.reserve(in_bytes, out_bytes);
    if (rc) return rc;
    cudaStream_t s = h->pipe.lane[0];
    CB_CUDA(cudaMemcpyAsync(h->pipe.in[0], in, in_bytes, cudaMemcpyHostToDevice, s));
    rc = cb_chain_run_dev(h, reinterpret_cast<const float *>(h->pipe.in[0]), n_in,
                          reinterpret_cast<float *>(h->pipe.out[0]), no, nullptr, s);
    if (rc) return rc;
    if (out_cap == no) {
        CB_CUDA(cudaMemcpyAsync(out, h->pipe.out[0], out_bytes, cudaMemcpyDeviceToHost, s));
    } else {  // caller's rows are out_cap apart
        const size_t esz = h->fm ? sizeof(float) : sizeof(float2);
        CB_CUDA(cudaMemcpy2DAsync(out, out_cap * esz, h->pipe.out[0], no * esz, no * esz, h->channels,
                                  cudaMemcpyDeviceToHost, s));
    }
    CB_CUDA(cudaStreamSynchronize(s));
    return CB_OK;
}

// ============================================================================ pulse-shaping taps
// rrc_taps (src/util/math.rs:221-280), host side, f64.
int cb_rrc_taps_f64(uint32_t n_taps, double sam_per_sym, double beta, double *taps)
{
    CB_REQUIRE(taps || n_taps == 0, CB_ERR_INVALID_ARG, "taps is NULL");
    CB_REQUIRE(beta >= 0.0 && beta <= 1.0, CB_ERR_INVALID_ARG, "rrc_taps: rolloff %g outside [0, 1]", beta);
    const double pi = 3.14159265358979323846, eps = 2.220446049250313e-16;
    const double at_zero = 1.0 + beta * (4.0 / pi - 1.0);
    const double at_sing = (beta / sqrt(2.0)) * ((1.0 + 2.0 / pi) * sin(pi / (4.0 * beta)) + (1.0 - 2.0 / pi) * cos(pi / (4.0 * beta)));
    const double t_sing = beta != 0.0 ? 1.0 / (4.0 * beta) : 0.0;
    for (uint32_t i = 0; i < n_taps; ++i) {
        const double t = ((double)i - (double)(n_taps - 1) / 2.0) / sam_per_sym;
        double v;
        if (fabs(t) < eps) {
            v = at_zero;
        } else if (fabs(t - t_sing) < eps || fabs(t + t_sing) < eps) {
            v = at_sing;
        } else {
            const double q = 4.0 * beta * t;
            v = (sin(pi * t * (1.0 - beta)) + 4.0 * beta * t * cos(pi * t * (1.0 + beta))) / (pi * t * (1.0 - q * q));
        }
        taps[2 * i] = v;
        taps[2 * i + 1] = 0.0;
    }
    return CB_OK;
}

int cb_rrc_taps(uint32_t n_taps, double sam_per_sym, double beta, float *taps)
{
    CB_REQUIRE(taps || n_taps == 0, CB_ERR_INVALID_ARG, "taps is NULL");
    std::vector<double> t((size_t)2 * n_taps);
    const int rc = cb_rrc_taps_f64(n_taps, sam_per_sym, beta, t.data());
    if (rc) return rc;
    for (size_t i = 0; i < t.size(); ++i) taps[i] = (float)t[i];
    return CB_OK;
}

// ============================================================================ f64 estimators (SURVEY 8(f) rank 2)
// qfilt_taps (src/util/math.rs:307-342), host side, f64: Mengali's q(t); an even n_taps is incremented by one.
int cb_qfilt_taps_f64(uint32_t n_taps, double alpha, uint32_t sam_per_sym, double *taps, uint32_t *n_out)
{
    CB_REQUIRE(alpha >= 0.0 && alpha <= 1.0, CB_ERR_INVALID_ARG, "qfilt_taps: rolloff %g outside [0, 1]", alpha);
    const uint32_t real_n = n_taps % 2 == 0 ? n_taps + 1 : n_taps;
    if (n_out) *n_out = real_n;
    CB_REQUIRE(taps, CB_ERR_INVALID_ARG, "taps is NULL");
    const double pi = 3.14159265358979323846;
    const int d = (int)floor((double)real_n / 2.0);
    for (uint32_t i = 0; i < real_n; ++i) {
        const double tt = (double)((int)i - d) / (double)sam_per_sym;
        const double two_alpha_tt = 2.0 * alpha * tt;
        if (fabs(two_alpha_tt) == 1.0) {
            taps[i] = sin(pi * alpha * tt) / (8.0 * tt);
        } else {
            taps[i] = (alpha * cos(pi * alpha * tt)) / (pi * (1.0 - two_alpha_tt * two_alpha_tt));
        }
    }
    return CB_OK;
}

// scratch of one estimator call, stream-ordered: partial sums, the final sum, optionally a staged copy of the samples
struct EstScratch {
    double2 *partial = nullptr, *sum = nullptr, *x = nullptr;
    cudaStream_t s = nullptr;
    int alloc(cudaStream_t stream, size_t n_stage)
    {
        s = stream;
        CB_CUDA(cudaMallocAsync(&partial, (estimator_max_partials() + 1) * sizeof(double2), s));
        sum = partial + estimator_max_partials();
        if (n_stage) CB_CUDA(cudaMallocAsync(&x, n_stage * sizeof(double2), s));
        return CB_OK;
    }
    ~EstScratch()
    {
        if (x) cudaFreeAsync(x, s);
        if (partial) cudaFreeAsync(partial, s);
    }
};

static int freq_estimate_impl(const double2 *samples, bool on_host, size_t n, double *estimate, cudaStream_t s)
{
    CB_REQUIRE(estimate, CB_ERR_INVALID_ARG, "estimate is NULL");
    if (n < 2) {  // empty sum: arg(0 + 0j) = 0
        *estimate = 0.0;
        return CB_OK;
    }
    CB_REQUIRE(samples, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE(on_host || (reinterpret_cast<uintptr_t>(samples) & 15) == 0, CB_ERR_INVALID_ARG,
               "frequency estimator: d_samples must be 16-byte aligned");  // read as double2
    int rc = ensure_device();
    if (rc) return rc;
    EstScratch sc;
    rc = sc.alloc(s, on_host ? n : 0);
    if (rc) return rc;
    if (on_host) CB_CUDA(cudaMemcpyAsync(sc.x, samples, n * sizeof(double2), cudaMemcpyHostToDevice, s));
    rc = launch_freq_sum(on_host ? sc.x : samples, n, sc.partial, sc.sum, s);
    if (rc) return rc;
    double2 sum;
    CB_CUDA(cudaMemcpyAsync(&sum, sc.sum, sizeof(sum), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
    *estimate = atan2(sum.y, sum.x);  // Complex::arg
    return CB_OK;
}

int cb_freq_estimate(const double *samples, size_t n, double *estimate)
{
    return freq_estimate_impl(reinterpret_cast<const double2 *>(samples), true, n, estimate, cudaStreamPerThread);
}

int cb_freq_estimate_dev(const double *d_samples, size_t n, double *estimate, void *stream)
{
    return freq_estimate_impl(reinterpret_cast<const double2 *>(d_samples), false, n, estimate,
                              stream ? (cudaStream_t)stream : cudaStreamPerThread);
}

struct cb_timing {
    int device;
    cudaStream_t stream;
    uint32_t n, d, ntaps;
    double *taps_dev;
};

int cb_timing_create(uint32_t n, uint32_t d, double alpha, cb_timing **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(n >= 1, CB_ERR_INVALID_ARG, "timing estimator: samples per symbol must be >= 1");
    CB_REQUIRE((uint64_t)2 * n * d + 1 <= 4097, CB_ERR_UNSUPPORTED,
               "timing estimator: filter length 2*n*d+1 = %llu > 4097 is not provided", (unsigned long long)2 * n * d + 1);
    int rc = ensure_device();
    if (rc) return rc;
    std::vector<double> taps((size_t)2 * n * d + 2);
    uint32_t ntaps = 0;
    rc = cb_qfilt_taps_f64(2 * n * d + 1, alpha, n, taps.data(), &ntaps);  // MathError::InvalidRolloffError
    if (rc) return rc;
    cb_timing *h = new (std::nothrow) cb_timing();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->stream = nullptr;
    h->n = n;
    h->d = d;
    h->ntaps = ntaps;
    h->taps_dev = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&h->taps_dev, ntaps * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(h->taps_dev, taps.data(), ntaps * sizeof(double), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cb_timing_destroy(h);
        return cuda_fail(e, "timing estimator create", __FILE__, __LINE__);
    }
    *out = h;
    return CB_OK;
}

int cb_timing_destroy(cb_timing *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->taps_dev) cudaFree(h->taps_dev);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

static int timing_push_impl(cb_timing *h, const double2 *samples, bool on_host, size_t n, double *estimate, cudaStream_t s)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(estimate, CB_ERR_INVALID_ARG, "estimate is NULL");
    const double pi = 3.14159265358979323846;
    double2 sum = make_double2(0.0, 0.0);
    if (n > 0) {
        CB_REQUIRE(samples, CB_ERR_INVALID_ARG, "NULL data pointer");
        CB_REQUIRE(on_host || (reinterpret_cast<uintptr_t>(samples) & 15) == 0, CB_ERR_INVALID_ARG,
                   "timing estimator: d_samples must be 16-byte aligned");  // read as double2
        CB_CUDA(cudaSetDevice(h->device));
        EstScratch sc;
        int rc = sc.alloc(s, on_host ? n : 0);
        if (rc) return rc;
        if (on_host) CB_CUDA(cudaMemcpyAsync(sc.x, samples, n * sizeof(double2), cudaMemcpyHostToDevice, s));
        rc = launch_timing_sum(on_host ? sc.x : samples, n, h->taps_dev, h->ntaps, h->n * h->d, h->n, sc.partial, sc.sum, s);
        if (rc) return rc;
        CB_CUDA(cudaMemcpyAsync(&sum, sc.sum, sizeof(sum), cudaMemcpyDeviceToHost, s));
        CB_CUDA(cudaStreamSynchronize(s));
    }
    *estimate = -(double)h->n * atan2(sum.y, sum.x) / (2.0 * pi);  // timing_estimator.rs:111
    return CB_OK;
}

int cb_timing_push(cb_timing *h, const double *samples, size_t n, double *estimate)
{
    return timing_push_impl(h, reinterpret_cast<const double2 *>(samples), true, n, estimate, h ? h->stream : nullptr);
}

int cb_timing_push_dev(cb_timing *h, const double *d_samples, size_t n, double *estimate, void *stream)
{
    return timing_push_impl(h, reinterpret_cast<const double2 *>(d_samples), false, n, estimate,
                            h ? pick_stream(stream, h->stream) : nullptr);
}

// ============================================================================ NCO (SURVEY 8(f) rank 4)
// Nco::new / Nco::push (src/demodulation/nco.rs:41-49, 71-77) and NcoNode::new(dphase, phase) (:112-127) over a batch
// of phase errors: out[k] = exp(j * phase_k), phase_k = phase_{k-1} + dphase + perr[k] (mod 2 pi), carried across calls.
struct cb_nco {
    int device;
    cudaStream_t stream;
    HostPipe pipe;
    double dphase;
    double *phase[2];
    int cur;
    double *scratch;
    size_t scratch_len;
    LastUse last;
};

int cb_nco_create(double dphase, double phase, cb_nco **out)
{
    CB_REQUIRE(out, CB_ERR_INVALID_ARG, "out is NULL");
    CB_REQUIRE(std::isfinite(dphase) && std::isfinite(phase), CB_ERR_INVALID_ARG, "nco: non-finite phase");
    int rc = ensure_device();
    if (rc) return rc;
    cb_nco *h = new (std::nothrow) cb_nco();
    CB_REQUIRE(h, CB_ERR_OOM, "host allocation failed");
    h->device = g_dev;
    h->dphase = wrap_dphase(dphase);  // the same wrap loop as Mixer::new (nco.rs:41-49)
    h->cur = 0;
    h->phase[0] = h->phase[1] = nullptr;
    h->scratch = nullptr;
    h->scratch_len = 0;
    h->stream = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaMalloc(&h->phase[i], sizeof(double));
        if (e == cudaSuccess) e = cudaMemcpy(h->phase[i], &phase, sizeof(double), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess || h->pipe.init(h->stream)) {
        cb_nco_destroy(h);
        return e != cudaSuccess ? cuda_fail(e, "nco create", __FILE__, __LINE__) : CB_ERR_CUDA;
    }
    *out = h;
    return CB_OK;
}

int cb_nco_destroy(cb_nco *h)
{
    if (!h) return CB_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->last.destroy();
    h->pipe.destroy();
    for (int i = 0; i < 2; ++i)
        if (h->phase[i]) cudaFree(h->phase[i]);
    if (h->scratch) cudaFree(h->scratch);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return CB_OK;
}

int cb_nco_run_dev(cb_nco *h, const double *d_perr, size_t n, double *d_out, void *stream)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_perr && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_REQUIRE((reinterpret_cast<uintptr_t>(d_out) & 15) == 0, CB_ERR_INVALID_ARG, "nco: d_out must be 16-byte aligned");
    CB_NO_ALIAS(d_perr, n * sizeof(double), d_out, n * 2 * sizeof(double), "nco");
    CB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = pick_stream(stream, h->stream);
    int rc = h->last.begin(s);
    if (rc) return rc;
    const size_t need = nco_scratch_doubles(n);
    if (h->scratch_len < need) {
        if (h->scratch) CB_CUDA(cudaFree(h->scratch));  // waits for earlier launches that use it
        h->scratch = nullptr;
        h->scratch_len = 0;
        CB_CUDA(cudaMalloc(&h->scratch, need * sizeof(double)));
        h->scratch_len = need;
    }
    rc = launch_nco(d_perr, n, h->scratch, h->phase[h->cur], h->phase[h->cur ^ 1], h->dphase,
                    reinterpret_cast<double2 *>(d_out), s);
    if (rc) return rc;
    h->cur ^= 1;
    return h->last.end(s);
}

int cb_nco_run(cb_nco *h, const double *perr, size_t n, double *out)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (n == 0) return CB_OK;
    CB_REQUIRE(perr && out, CB_ERR_INVALID_ARG, "NULL data pointer");
    CB_CUDA(cudaSetDevice(h->device));
    int rc = h->pipe.reserve(n * sizeof(double), n * 2 * sizeof(double));
    if (rc) return rc;
    cudaStream_t s = h->pipe.lane[0];
    CB_CUDA(cudaMemcpyAsync(h->pipe.in[0], perr, n * sizeof(double), cudaMemcpyHostToDevice, s));
    rc = cb_nco_run_dev(h, reinterpret_cast<const double *>(h->pipe.in[0]), n, reinterpret_cast<double *>(h->pipe.out[0]), s);
    if (rc) return rc;
    CB_CUDA(cudaMemcpyAsync(out, h->pipe.out[0], n * 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
    CB_CUDA(cudaStreamSynchronize(s));
    return CB_OK;
}

int cb_nco_get_phase(cb_nco *h, double *phase, double *dphase)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    if (dphase) *dphase = h->dphase;
    if (phase) {
        CB_CUDA(cudaSetDevice(h->device));
        CB_CUDA(cudaStreamSynchronize(h->stream));
        int rc = h->last.sync();
        if (rc) return rc;
        CB_CUDA(cudaMemcpy(phase, h->phase[h->cur], sizeof(double), cudaMemcpyDeviceToHost));
    }
    return CB_OK;
}

int cb_nco_set_phase(cb_nco *h, double phase)
{
    CB_REQUIRE(h, CB_ERR_INVALID_ARG, "handle is NULL");
    CB_REQUIRE(std::isfinite(phase), CB_ERR_INVALID_ARG, "nco: non-finite phase");
    CB_CUDA(cudaSetDevice(h->device));
    CB_CUDA(cudaStreamSynchronize(h->stream));
    int rc = h->last.sync();
    if (rc) return rc;
    CB_CUDA(cudaMemcpy(h->phase[h->cur], &phase, sizeof(double), cudaMemcpyHostToDevice));
    return CB_OK;
}

// ============================================================================ bit-exact edges
int cb_prn_bits(uint64_t poly_mask, uint64_t *state, unsigned width, size_t n, uint8_t *bits)
{
    // PrnGen::next_byte (src/prns.rs:64-71); a serial recurrence, evaluated on the host.
    CB_REQUIRE(state && (bits || n == 0), CB_ERR_INVALID_ARG, "NULL argument");
    CB_REQUIRE(width == 8 || width == 16 || width == 32 || width == 64, CB_ERR_INVALID_ARG,
               "prn: register width must be 8, 16, 32 or 64");
    const uint64_t wm = width >= 64 ? ~0ULL : ((1ULL << width) - 1ULL);
    uint64_t st = *state & wm;
    for (size_t i = 0; i < n; ++i) {
        const uint64_t fb = (uint64_t)(__builtin_popcountll(st & poly_mask & wm) & 1);
        bits[i] = (uint8_t)(st >> (width - 1));
        st = ((st << 1) & wm) | fb;
    }
    *state = st;
    return CB_OK;
}

int cb_bits_to_symbols_dev(const uint8_t *d_bits, size_t nbits, int mode, float *d_sym, size_t *nsym, void *stream)
{
    CB_REQUIRE(mode == 0 || mode == 1, CB_ERR_INVALID_ARG, "bits_to_symbols: mode must be 0 (BPSK) or 1 (QPSK)");
    const size_t ns = mode == 0 ? nbits : nbits / 2;
    if (nsym) *nsym = ns;
    if (ns == 0) return CB_OK;
    CB_REQUIRE(d_bits && d_sym, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_bits_to_symbols(d_bits, reinterpret_cast<float2 *>(d_sym), ns, mode, (cudaStream_t)stream);
}

int cb_real_to_complex_dev(const float *d_in, size_t n, float *d_out, void *stream)
{
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_real_to_complex(d_in, reinterpret_cast<float2 *>(d_out), n, (cudaStream_t)stream);
}

int cb_complex_real_dev(const float *d_in, size_t n, float *d_out, void *stream)
{
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_complex_real(reinterpret_cast<const float2 *>(d_in), d_out, n, (cudaStream_t)stream);
}

int cb_convert_u8_dev(const uint8_t *d_in, size_t n_samples, float *d_out, void *stream)
{
    if (n_samples == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_convert_u8(d_in, d_out, 2 * n_samples, (cudaStream_t)stream);
}

int cb_convert_i16_dev(const int16_t *d_in, size_t n_samples, float scale, float *d_out, void *stream)
{
    if (n_samples == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_convert_i16(d_in, d_out, 2 * n_samples, scale, (cudaStream_t)stream);
}

int cb_quantize_i16_dev(const float *d_in, size_t nfloats, float scale, int16_t *d_out, void *stream)
{
    if (nfloats == 0) return CB_OK;
    CB_REQUIRE(d_in && d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_quantize_i16(d_in, d_out, nfloats, scale, (cudaStream_t)stream);
}

int cb_synth_uniform_dev(uint64_t seed, uint64_t first, size_t n, float *d_out, void *stream)
{
    if (n == 0) return CB_OK;
    CB_REQUIRE(d_out, CB_ERR_INVALID_ARG, "NULL data pointer");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_synth(d_out, 2 * n, seed + 2 * first, (cudaStream_t)stream);
}

}  // extern "C"
