// Shared declarations of the metric-suite kernels (reference core/metric.py).
#pragma once
#include "moment_fwd.cuh"

namespace mmif {

constexpr int kPixelMinRows = 8;  // smallest row chunk of a stats / Qabf CTA (workspace sizing)
constexpr int kRawPerPair = 160;   // doubles of raw per-pair results inside the workspace

// Workspace carve-up (all device memory owned by the caller, see mmif_metric_workspace_bytes).
struct MetricWs {
    unsigned* counters;     // [N+1], zero between launches
    double* partial;        // per-CTA partial sums of the simple kernels
    unsigned char* fwd_ws;  // counters + partials of the strip-streaming kernel
    size_t fwd_ws_bytes;
    uint32_t* hist_extra;   // [hist_extra_words(N)], zero between launches
    double* raw;            // [N][kRawPerPair]
    float* pyr;             // pyramid levels (MS-SSIM) / decimated scales (VIF)
    size_t pyr_floats;
    uint32_t* counts;       // [N][MMIF_HIST_WORDS] histogram block used by mmif_eval_suite
    unsigned char* fwd_ws_b; // second strip-kernel workspace + pyramid: the VIF chain of mmif_eval_suite runs
    float* pyr_b;            // concurrently with the MS-SSIM chain (forked streams)
};
size_t metric_ws_bytes(int N, int H, int W);
int carve_metric_ws(MetricWs* w, void* ws, size_t ws_bytes, int N, int H, int W);

// raw[] layout per pair
enum {
    RAW_STATS = 0,          // MMIF_ST_COUNT (16)
    RAW_ENT = 16,           // MMIF_EN_COUNT (12)
    RAW_QABF = 28,          // 4
    RAW_SSIM = 32,          // 8 raw sums of the 11-tap SSIM kernel (level 0)
    RAW_MS = 40,            // 5 levels x 8
    RAW_VIF = 80,           // 4 scales x 8
    RAW_SSIM_OUT = 112,     // 4
    RAW_MS_OUT = 116,       // MMIF_MSSSIM_DOUBLES (22)
    RAW_VIF_OUT = 138       // up to 160: viff, viff_simple (+ per-scale sums live in RAW_VIF)
};

int launch_stats(const float* a, const float* b, const float* f, int N, int H, int W, double* out, long long ostride, MetricWs& ws,
                 cudaStream_t st);
int launch_stats_bwd(const float* a, const float* b, const float* f, int N, int H, int W, const double* row, const float* gout,
                     float* da, float* db, float* df, cudaStream_t st);
int launch_hist(const float* a, const float* b, const float* f, int N, int H, int W, uint32_t* counts, double* ent,
                long long estride, MetricWs& ws, cudaStream_t st);
int launch_qabf(const float* a, const float* b, const float* f, int N, int H, int W, float L, double* out, long long ostride,
                MetricWs& ws, cudaStream_t st, int q_raw = 0);
int launch_pixel_metrics(const float* a, const float* b, const float* f, int N, int H, int W, float L, double* out_s,
                         long long sstride, double* out_q, long long qstride, MetricWs& ws, cudaStream_t st, int q_raw = 0);
int launch_tv(const float* x, int N, int H, int W, int norm, float weight, double* out, MetricWs& ws, cudaStream_t st);
int stats_rows_per_block(int N, int H);
size_t hist_extra_words(int N);

#ifdef __CUDACC__
// Block partial -> global; the last block of sample n re-reduces all partials of that sample in a
// fixed order.  Returns true on thread 0 of that last block only, with the totals in t[].
template <int K, int NTHREADS>
__device__ __forceinline__ bool block_finish(double (&v)[K], double* red, int* flag, double* partial, unsigned* counters,
                                             int n, int blk, int nblk, double (&t)[K]) {
    block_sum<K, NTHREADS>(v, red);
    if (threadIdx.x == 0) {
        double* dst = partial + ((size_t)n * nblk + blk) * K;
#pragma unroll
        for (int i = 0; i < K; ++i) dst[i] = v[i];
        __threadfence();
        const unsigned prev = atomicAdd(&counters[n], 1u);
        *flag = (prev == (unsigned)(nblk - 1));
    }
    __syncthreads();
    if (!*flag) return false;
    __threadfence();
#pragma unroll
    for (int i = 0; i < K; ++i) t[i] = 0.0;
    for (int k = threadIdx.x; k < nblk; k += NTHREADS) {
        const double* src = partial + ((size_t)n * nblk + k) * K;
#pragma unroll
        for (int i = 0; i < K; ++i) t[i] += __ldcg(src + i);
    }
    block_sum<K, NTHREADS>(t, red);
    if (threadIdx.x == 0) counters[n] = 0u;
    return threadIdx.x == 0;
}
#endif

}  // namespace mmif
