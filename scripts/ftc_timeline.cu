// Phase sums of the tensor-core FIR (fir_tc_kernel.cu, K1-TC): compiled with CB_FTC_STATS, clock64 sums per phase over
// every tile of a CTA, one thread of each role (TMA warp, the two converter groups, MMA warp, epilogue warp 0).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o /tmp/ftc_timeline scripts/ftc_timeline.cu
//   /tmp/ftc_timeline [log2 samples] [taps] [iq16: 0 | 1] [random data: 0 | 1]
#define CB_FTC_STATS
#include <cstdarg>
#include <cmath>
#include <algorithm>
#include <vector>
#include "../comms-rs_b200/csrc/fir_tc_kernel.cu"

namespace cb {
void set_error(const char *fmt, ...) { va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap); fputc('\n', stderr); }
int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    fprintf(stderr, "%s:%d %s: %s\n", file, line, what, cudaGetErrorString(e));
    return CB_ERR_CUDA;
}
void count_launch() {}
int launch_fir_fixup(const FirFixArgs &, cudaStream_t) { return CB_OK; }
}  // namespace cb

__global__ void fill_hash(unsigned *p, size_t n, int iq16)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned h = (unsigned)i * 2654435761u;
        h ^= h >> 15;
        h *= 2246822519u;
        h ^= h >> 13;
        // f32: sign + exponent of [0.5, 1) + random mantissa; i16: any word
        p[i] = iq16 ? h : ((h & 0x807fffffu) | 0x3f000000u);
    }
}

int main(int argc, char **argv)
{
    const size_t n = (size_t)1 << (argc > 1 ? atoi(argv[1]) : 28);
    const unsigned ntaps = argc > 2 ? atoi(argv[2]) : 64;
    const bool iq16 = argc > 3 && atoi(argv[3]) != 0;
    const unsigned H = 128;
    float2 *x, *y, *hist[2];
    cudaMalloc(&x, n * 8);
    cudaMalloc(&y, n * 8);
    if (argc > 4 && atoi(argv[4]) != 0) fill_hash<<<148 * 8, 256>>>(reinterpret_cast<unsigned *>(x), n * 2, iq16);  // random samples
    else cudaMemset(x, 0x3c, n * 8);  // constant, finite, non-zero words in either format
    for (int i = 0; i < 2; ++i) {
        cudaMalloc(&hist[i], H * 8);
        cudaMemset(hist[i], 0, H * 8);
    }
    std::vector<float2> taps(ntaps);
    for (unsigned k = 0; k < ntaps; ++k) taps[k] = make_float2((float)std::cos(0.1 * k) / (1 + k), (float)std::sin(0.3 * k) / (2 + k));
    std::vector<unsigned char> himg(cb::fir_tc_image_bytes(ntaps));
    float tis = 1.f;
    cb::fir_tc_build_image(taps.data(), ntaps, himg.data(), &tis);
    unsigned char *img;
    cudaMalloc(&img, himg.size());
    cudaMemcpy(img, himg.data(), himg.size(), cudaMemcpyHostToDevice);
    unsigned long long *dbg;
    const size_t ncta = 148;
    cudaMalloc(&dbg, ncta * 5 * 8 * 8);
    cudaMemset(dbg, 0, ncta * 5 * 8 * 8);
    cudaMemcpyToSymbol(cb::tc::g_ftc_dbg, &dbg, sizeof(dbg));
    cb::FirSeg seg{x, hist[0], hist[1], y, n, n, H, ntaps, 1, 1};
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    for (int it = 0; it < 3; ++it) {
        cudaEventRecord(e0);
        const cb::FirTcPlan plan{img, tis, 1};
        int rc = iq16 ? cb::launch_fir_tc_iq16(seg, reinterpret_cast<const int16_t *>(x), 1.f / 32768, reinterpret_cast<int16_t *>(y), 8192.f, plan, nullptr, 0)
                      : cb::launch_fir_tc(seg, plan, nullptr, 0);
        if (rc) return 1;
        cudaEventRecord(e1);
        if (cudaDeviceSynchronize() != cudaSuccess) { fprintf(stderr, "kernel failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 1; }
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        printf("run %d: %.4f ms  %.1f Gsamples/s\n", it, ms, n / ms / 1e6);
    }
    std::vector<unsigned long long> d(ncta * 5 * 8);
    cudaMemcpy(d.data(), dbg, d.size() * 8, cudaMemcpyDeviceToHost);
    const size_t tiles = (n + 4095) / 4096;
    const char *role[5] = {"TMA warp", "converter group 0 (even tiles)", "converter group 1 (odd tiles)", "MMA warp", "epilogue warp 0"};
    const char *ph[5][8] = {
        {"issue copies + loop", "wait raw_empty (converters have read the stage)", 0, 0, 0, 0, 0, 0},
        {"flagging + loop", "wait raw_full (TMA landed)", "load raw + max/min", "group barrier", "scale exponent", "wait a_empty (MMAs done with the stage)", "scale, split, st.shared, fence, arrive", 0},
        {"flagging + loop", "wait raw_full (TMA landed)", "load raw + max/min", "group barrier", "scale exponent", "wait a_empty (MMAs done with the stage)", "scale, split, st.shared, fence, arrive", 0},
        {"issue MMAs + commit", "wait t_empty (epilogue has drained the accumulator)", "wait a_full (converters)", 0, 0, 0, 0, 0},
        {"loop", "wait sc_ready + t_full (MMAs done)", "tcgen05.ld, unscale, store", 0, 0, 0, 0, 0}};
    for (int r = 0; r < 5; ++r) {
        double sum[8] = {0}, tot = 0;
        for (size_t c = 0; c < ncta; ++c)
            for (int k = 0; k < 8; ++k) sum[k] += (double)d[(c * 5 + r) * 8 + k];
        for (int k = 0; k < 8; ++k) tot += sum[k];
        const double per = (r == 1 || r == 2) ? tiles / 2.0 : (double)tiles;
        printf("%s: %.0f cycles per tile it handles\n", role[r], tot / per);
        for (int k = 0; k < 8; ++k)
            if (ph[r][k]) printf("   %5.1f %%  %6.0f cyc  %s\n", 100 * sum[k] / tot, sum[k] / per, ph[r][k]);
    }
    return 0;
}
