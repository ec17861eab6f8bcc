// Structural-similarity and visual-information-fidelity families of reference core/metric.py
// (calc_ssim :316-364, calc_msssim :368-402, calc_vif :406-458, calc_viff :461-491), the 16-metric
// row of eval.py:29-75, and the C ABI entry points of the metric suite.
#include <stdlib.h>
#include "metrics.cuh"

namespace mmif {

static inline size_t al256(size_t v) { return (v + 255) / 256 * 256; }

// =============================================================================== small generic SSIM
// Any window size k <= 11 (metric.py:323-325 shrinks the window to min(win, H, W) for tiny images,
// e.g. the deepest MS-SSIM levels): one thread per window position, the k x k float32 window
// W[i][j] = fl(w_i * w_j) exactly as torch.mm builds it, moments accumulated in double.
__global__ void __launch_bounds__(256)
ssim_small_kernel(const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ F, int H, int W, int k,
                  const Taps taps, double C1, double C2, double* partial, unsigned* counters, double* sums, long long stride) {
    __shared__ double red[8 * 8];
    __shared__ int flag;
    const int n = blockIdx.y, blk = blockIdx.x, nblk = gridDim.x;
    const int Ho = H - k + 1, Wo = W - k + 1;
    const size_t off = (size_t)n * H * W;
    const float* a = A + off; const float* b = Bm + off; const float* f = F + off;
    double acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0;
    const long long idx = (long long)blk * 256 + threadIdx.x;
    if (idx < (long long)Ho * Wo) {
        const int i0 = (int)(idx / Wo), j0 = (int)(idx % Wo);
        double m1 = 0, m2 = 0, mf = 0, e11 = 0, e22 = 0, eff = 0, e1f = 0, e2f = 0;
        for (int u = 0; u < k; ++u)
            for (int v = 0; v < k; ++v) {
                const double w = (double)(float)(taps.w[u] * taps.w[v]);
                const size_t p = (size_t)(i0 + u) * W + (j0 + v);
                const double x1 = a[p], x2 = b[p], y = f[p];
                m1 += w * x1; m2 += w * x2; mf += w * y;
                e11 += w * x1 * x1; e22 += w * x2 * x2; eff += w * y * y;
                e1f += w * x1 * y; e2f += w * x2 * y;
            }
        const double vf = fmax(eff - mf * mf, 0.0);
        const double mk[2] = {m1, m2}, ek[2] = {e11, e22}, ekf[2] = {e1f, e2f};
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const double vk = fmax(ek[s] - mk[s] * mk[s], 0.0);
            const double cov = ekf[s] - mk[s] * mf;
            const double A1 = 2.0 * mk[s] * mf + C1, B1 = mk[s] * mk[s] + mf * mf + C1;
            const double A2 = 2.0 * cov + C2, B2 = vk + vf + C2;
            acc[0 + s] = (A1 * A2) / (B1 * B2);
            acc[2 + s] = A2 / B2;
            acc[4 + s] = fmax(vk, 1e-4);
        }
    }
    double t[8];
    if (!block_finish<8, 256>(acc, red, &flag, partial, counters, n, blk, nblk, t)) return;
    double* d = sums + (size_t)n * stride;
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = t[i];
}

// SSIM raw sums of the pairs (a,f), (b,f) at one pyramid level -> sums[n*stride + 0..7].
static int run_ssim_level(const float* a, const float* b, const float* f, int N, int H, int W, int win_size, float data_range,
                          double* sums, long long stride, MetricWs& ws, cudaStream_t st) {
    const int k = win_size < H ? (win_size < W ? win_size : W) : (H < W ? H : W);
    if (k == 11) {
        FwdLaunch L;
        memset(&L, 0, sizeof(L));
        L.win = 11; L.sigma = 1.5; L.epi = EPI_SSIM; L.finalize = FIN_SUMS; L.do_sobel = 0; L.data_range = data_range;
        L.cfg.pixel_norm = L.cfg.grad_norm = MMIF_NORM_L1;
        return launch_moment_fwd(L, a, b, f, N, H, W, sums, stride, nullptr, ws.fwd_ws, ws.fwd_ws_bytes, st);
    }
    if (k < 1 || k > 11) { set_error("ssim: window %d unsupported (1..11)", k); return MMIF_E_MODE; }
    Taps taps;
    make_taps(&taps, k, 1.5);
    const double R = data_range;
    const long long npos = (long long)(H - k + 1) * (W - k + 1);
    dim3 grid((unsigned)((npos + 255) / 256), N);
    // The deep pyramid levels (image smaller than the window) keep counters + partials in the chain's own
    // strip-kernel workspace: the chains of mmif_eval_suite run concurrently and the shared ws.partial
    // belongs to the pixel kernel there.  A small window on a large image (mmif_ssim only) uses ws.partial.
    const size_t small_need = ws_counters_bytes(N) + (size_t)N * grid.x * 8 * sizeof(double);
    double* part = ws.partial; unsigned* cnt = ws.counters;
    if (small_need <= ws.fwd_ws_bytes) { part = (double*)(ws.fwd_ws + ws_counters_bytes(N)); cnt = (unsigned*)ws.fwd_ws; }
    ssim_small_kernel<<<grid, 256, 0, st>>>(a, b, f, H, W, k, taps, (0.01 * R) * (0.01 * R), (0.03 * R) * (0.03 * R), part, cnt,
                                            sums, stride);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// =============================================================================== pyramid steps
// MS-SSIM level step (metric.py:389-395): reflect-pad the odd edge, 2x2 mean.  ATen's avg_pool2d
// adds the window in row-major order and divides by 4.  One output per thread; each thread reads
// two float2 (coalesced 8-byte loads) when the row pitch allows.
struct Ptr3 { const float* src[3]; float* dst[3]; };
__global__ void __launch_bounds__(256) halve_kernel(Ptr3 p, int N, int H, int W, int Ho, int Wo) {
    const int k = blockIdx.z % 3, n = blockIdx.z / 3;
    const int j = blockIdx.x * 64 + (threadIdx.x & 63);
    const int i = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (i >= Ho || j >= Wo) return;
    const float* s = p.src[k] + (size_t)n * H * W;
    const int r0 = 2 * i, r1 = (2 * i + 1 < H) ? 2 * i + 1 : H - 2;
    const int c0 = 2 * j, c1 = (2 * j + 1 < W) ? 2 * j + 1 : W - 2;
    float a, b, c, d;
    if ((W & 1) == 0 && (((uintptr_t)s) & 7) == 0) {
        const float2 t0 = __ldg(reinterpret_cast<const float2*>(s + (size_t)r0 * W + c0));
        const float2 t1 = __ldg(reinterpret_cast<const float2*>(s + (size_t)r1 * W + c0));
        a = t0.x; b = t0.y; c = t1.x; d = t1.y;
    } else {
        a = __ldg(s + (size_t)r0 * W + c0); b = __ldg(s + (size_t)r0 * W + c1);
        c = __ldg(s + (size_t)r1 * W + c0); d = __ldg(s + (size_t)r1 * W + c1);
    }
    p.dst[k][((size_t)n * Ho + i) * Wo + j] = (((a + b) + c) + d) * 0.25f;
}

// Same step when the row pitch allows 16-byte loads (W % 4 == 0, so no odd-column pad): one thread =
// 2 x 2 outputs from four float4 loads (64 B in flight per thread), the odd bottom row reflected.
__global__ void __launch_bounds__(256) halve4_kernel(Ptr3 p, int N, int H, int W, int Ho, int Wo) {
    const int k = blockIdx.z % 3, n = blockIdx.z / 3;
    const int j2 = blockIdx.x * 32 + (threadIdx.x & 31);          // pair of output columns
    const int i2 = blockIdx.y * 8 + (threadIdx.x >> 5);           // pair of output rows
    if (2 * j2 >= Wo || 2 * i2 >= Ho) return;
    const float* s = p.src[k] + (size_t)n * H * W + 4 * j2;
    float* d = p.dst[k] + ((size_t)n * Ho + 2 * i2) * Wo + 2 * j2;
    const int r0 = 4 * i2;
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(s + (size_t)r0 * W));
    const float4 a1 = __ldg(reinterpret_cast<const float4*>(s + (size_t)((r0 + 1 < H) ? r0 + 1 : H - 2) * W));
    *reinterpret_cast<float2*>(d) = make_float2((((a0.x + a0.y) + a1.x) + a1.y) * 0.25f, (((a0.z + a0.w) + a1.z) + a1.w) * 0.25f);
    if (2 * i2 + 1 < Ho) {
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(s + (size_t)(r0 + 2) * W));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(s + (size_t)((r0 + 3 < H) ? r0 + 3 : H - 2) * W));
        *reinterpret_cast<float2*>(d + Wo) = make_float2((((b0.x + b0.y) + b1.x) + b1.y) * 0.25f, (((b0.z + b0.w) + b1.z) + b1.w) * 0.25f);
    }
}
static int launch_halve(const Ptr3& p, int N, int H, int W, int Ho, int Wo, cudaStream_t st) {
    bool vec = (W % 4 == 0);
    for (int k = 0; k < 3; ++k) vec = vec && ((((uintptr_t)p.src[k]) & 15) == 0) && ((((uintptr_t)p.dst[k]) & 7) == 0);
    if (vec) {
        dim3 grid(ceil_div(Wo, 64), ceil_div(Ho, 16), 3 * N);
        halve4_kernel<<<grid, 256, 0, st>>>(p, N, H, W, Ho, Wo);
        mmif::count_launch(MMIF_CNT_METRIC);
    } else {
        dim3 grid(ceil_div(Wo, 64), ceil_div(Ho, 4), 3 * N);
        halve_kernel<<<grid, 256, 0, st>>>(p, N, H, W, Ho, Wo);
        mmif::count_launch(MMIF_CNT_METRIC);
    }
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// VIF scale step (metric.py:419-423): valid K x K Gaussian blur, then every other row / column.
// thread = output column, marching down a segment of output rows: each input row is blurred
// horizontally at the even columns straight from global memory (K contiguous values per thread, 8-byte
// loads when the pitch allows; a warp covers 64+K-1 contiguous floats per row, the re-reads hit L1), the
// last K horizontal results slide through registers and every second row emits one vertical blur:
// 3K/4 FMA per input pixel, each input read from DRAM once.
constexpr int kBdRows = 32;      // output rows per CTA
template <int K, bool VEC>
__device__ __forceinline__ float hblur_row(const float* __restrict__ q, const Taps& taps) {
    float acc = 0.f;
    if (VEC) {
#pragma unroll
        for (int v = 0; v + 1 < K; v += 2) {
            const float2 x = __ldg(reinterpret_cast<const float2*>(q + v));
            acc = fmaf(taps.w[v], x.x, acc);
            acc = fmaf(taps.w[v + 1], x.y, acc);
        }
        acc = fmaf(taps.w[K - 1], __ldg(q + K - 1), acc);      // K is odd
    } else {
#pragma unroll
        for (int v = 0; v < K; ++v) acc = fmaf(taps.w[v], __ldg(q + v), acc);
    }
    return acc;
}
template <int K, bool VEC>
__global__ void __launch_bounds__(128) blur_decimate_kernel(Ptr3 p, int N, int H, int W, int Ho, int Wo, const __grid_constant__ Taps taps) {
    const int im = blockIdx.z % 3, n = blockIdx.z / 3;
    const int j = blockIdx.x * 128 + threadIdx.x;
    if (j >= Wo) return;
    const int oi0 = blockIdx.y * kBdRows, oi1 = min(oi0 + kBdRows, Ho);
    const float* q = p.src[im] + (size_t)n * H * W + (size_t)(2 * oi0) * W + 2 * j;
    float* dst = p.dst[im] + ((size_t)n * Ho + oi0) * Wo + j;
    float h[K];                                  // horizontal blurs of input rows 2*oi .. 2*oi + K-1
#pragma unroll
    for (int u = 0; u < K - 2; ++u) h[u + 2] = hblur_row<K, VEC>(q + (size_t)u * W, taps);
    q += (size_t)(K - 2) * W;
    for (int oi = oi0; oi < oi1; ++oi) {
#pragma unroll
        for (int u = 0; u < K - 2; ++u) h[u] = h[u + 2];
        h[K - 2] = hblur_row<K, VEC>(q, taps);
        h[K - 1] = hblur_row<K, VEC>(q + W, taps);
        q += 2 * (size_t)W;
        float acc = 0.f;
#pragma unroll
        for (int u = 0; u < K; ++u) acc = fmaf(taps.w[u], h[u], acc);
        *dst = acc;
        dst += Wo;
    }
}
template <int K>
static int launch_bd(const Ptr3& p, int N, int H, int W, int Ho, int Wo, const Taps& taps, cudaStream_t st) {
    dim3 grid(ceil_div(Wo, 128), ceil_div(Ho, kBdRows), 3 * N);
    const bool vec = ((W & 1) == 0) && ((((uintptr_t)p.src[0] | (uintptr_t)p.src[1] | (uintptr_t)p.src[2]) & 7) == 0);
    if (vec) blur_decimate_kernel<K, true><<<grid, 128, 0, st>>>(p, N, H, W, Ho, Wo, taps);
    else blur_decimate_kernel<K, false><<<grid, 128, 0, st>>>(p, N, H, W, Ho, Wo, taps);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// =============================================================================== compose kernels
struct LevelDims { int h[5], w[5], k[5]; };

__global__ void ssim_out_kernel(const double* raw, long long stride, int N, double inv, double* out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const double* s = raw + (size_t)n * stride;
    double* o = out + (size_t)n * 4;
    o[0] = s[0] * inv; o[1] = s[2] * inv; o[2] = s[1] * inv; o[3] = s[3] * inv;   // ssim_af, cs_af, ssim_bf, cs_bf
}

__device__ __forceinline__ void msssim_of(const double* ms /*5 x 8 raw*/, const LevelDims& d, double* o /*22*/) {
    const double wts[5] = {(double)0.0448f, (double)0.2856f, (double)0.3001f, (double)0.2363f, (double)0.1333f};
    double prod[2] = {1.0, 1.0};
    for (int l = 0; l < 5; ++l) {
        const double inv = 1.0 / ((double)(d.h[l] - d.k[l] + 1) * (double)(d.w[l] - d.k[l] + 1));
        const double* s = ms + l * 8;
        const double ssim[2] = {s[0] * inv, s[1] * inv}, cs[2] = {s[2] * inv, s[3] * inv};
        o[2 + l * 4 + 0] = ssim[0]; o[2 + l * 4 + 1] = cs[0]; o[2 + l * 4 + 2] = ssim[1]; o[2 + l * 4 + 3] = cs[1];
        for (int k = 0; k < 2; ++k) {
            const double v = fmax(l < 4 ? cs[k] : ssim[k], 1e-7);      // metric.py:386-399
            prod[k] *= pow(v, wts[l]);
        }
    }
    o[0] = prod[0]; o[1] = prod[1];
}
__global__ void msssim_out_kernel(const double* raw, long long stride, int N, LevelDims d, double* out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    msssim_of(raw + (size_t)n * stride, d, out + (size_t)n * MMIF_MSSSIM_DOUBLES);
}

__device__ __forceinline__ void viff_of(const double* vs /*4 x 8 raw*/, double* o /*26*/) {
    const double p[4] = {(double)(1.0f / 2.15f), (double)(0.0f / 2.15f), (double)(0.15f / 2.15f), (double)(1.0f / 2.15f)};
    double full = 0.0, n1 = 0.0, d1 = 0.0, n2 = 0.0, d2 = 0.0;
    for (int s = 0; s < 4; ++s) {
        const double* q = vs + s * 8;     // num1, den1, num2, den2, numsel, densel
        for (int i = 0; i < 6; ++i) o[2 + s * 6 + i] = q[i];
        full += p[s] * (double)(float)(q[4] / q[5]);     // viff[i] is stored in a float32 tensor (metric.py:479,489)
        n1 += q[0]; d1 += q[1]; n2 += q[2]; d2 += q[3];
    }
    o[0] = full;
    o[1] = n1 / d1 + n2 / d2;
}
__global__ void viff_out_kernel(const double* raw, long long stride, int N, double* out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    viff_of(raw + (size_t)n * stride, out + (size_t)n * MMIF_VIFF_DOUBLES);
}

// eval.py:29-75 row: sd ag sf mse psnr cc scd en ce mi qabf nabf labf ssim msssim viff
__global__ void suite_out_kernel(const double* raw, int N, LevelDims d, double inv_ssim, double* out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const double* r = raw + (size_t)n * kRawPerPair;
    const double* st = r + RAW_STATS; const double* en = r + RAW_ENT; const double* q = r + RAW_QABF;
    double* o = out + (size_t)n * MMIF_EVAL_METRICS;
    o[0] = st[MMIF_ST_SD]; o[1] = st[MMIF_ST_AG]; o[2] = st[MMIF_ST_SF];
    const double mse = (st[MMIF_ST_MSE_AF] + st[MMIF_ST_MSE_BF]) * 0.5;
    o[3] = mse; o[4] = 10.0 * log10(1.0 / mse);                               // calc_psnr(mse), metric.py:72-76
    o[5] = (st[MMIF_ST_CC_AF] + st[MMIF_ST_CC_BF]) * 0.5; o[6] = st[MMIF_ST_SCD];
    o[7] = en[MMIF_EN_F]; o[8] = en[MMIF_CE_AF] + en[MMIF_CE_BF]; o[9] = en[MMIF_NMI_AF] + en[MMIF_NMI_BF];
    o[10] = q[0]; o[11] = q[1]; o[12] = q[2];
    const double* s = r + RAW_MS;     // level 0 of the pyramid = the plain 11-tap SSIM
    o[13] = (s[0] * inv_ssim + s[1] * inv_ssim) * 0.5;
    double ms[MMIF_MSSSIM_DOUBLES], vf[MMIF_VIFF_DOUBLES];
    msssim_of(r + RAW_MS, d, ms);
    o[14] = (ms[0] + ms[1]) * 0.5;
    viff_of(r + RAW_VIF, vf);
    o[15] = vf[0];
}

// =============================================================================== drivers
static LevelDims msssim_dims(int H, int W, int win) {
    LevelDims d;
    int h = H, w = W;
    for (int l = 0; l < 5; ++l) {
        d.h[l] = h; d.w[l] = w;
        d.k[l] = win < h ? (win < w ? win : w) : (h < w ? h : w);
        h = (h + (h & 1)) / 2; w = (w + (w & 1)) / 2;
    }
    return d;
}
static size_t msssim_pyr_floats(int N, int H, int W) {
    const LevelDims d = msssim_dims(H, W, 11);
    size_t t = 0;
    for (int l = 1; l < 5; ++l) t += (size_t)3 * N * d.h[l] * d.w[l];
    return t;
}
static const int kVifWin[4] = {17, 9, 5, 3};
struct VifDims { int h[4], w[4]; bool ok; };
static VifDims vif_dims(int H, int W) {
    VifDims d;
    d.ok = true;
    int h = H, w = W;
    for (int s = 0; s < 4; ++s) {
        const int k = kVifWin[s];
        if (s > 0) {
            if (h < k || w < k) { d.ok = false; h = w = 1; }
            else { h = (h - k + 2) / 2; w = (w - k + 2) / 2; }
        }
        d.h[s] = h; d.w[s] = w;
        if (h < k || w < k) d.ok = false;
    }
    return d;
}
static size_t vif_pyr_floats(int N, int H, int W) {
    const VifDims d = vif_dims(H, W);
    size_t t = 0;
    for (int s = 1; s < 4; ++s) t += (size_t)3 * N * d.h[s] * d.w[s];
    return t;
}

size_t metric_ws_bytes(int N, int H, int W) {
    if (N < 1 || H < 1 || W < 1) return 0;
    size_t partial = (size_t)N * ceil_div(H, stats_rows_per_block(N, H)) * 14;
    const size_t pq = (size_t)N * ceil_div(W, 128) * ceil_div(H, kPixelMinRows) * 19;
    const size_t ps = (size_t)N * (((size_t)H * W + 255) / 256) * 8;
    partial = partial > pq ? partial : pq;
    partial = partial > ps ? partial : ps;
    size_t fwd = 0;
    const LevelDims md = msssim_dims(H, W, 11);
    for (int l = 0; l < 5; ++l) {
        size_t b = fwd_ws_bytes(11, N, md.h[l], md.w[l]);
        if (md.k[l] < 11) b = ws_counters_bytes(N) + (size_t)N * (((size_t)md.h[l] * md.w[l] + 255) / 256) * 8 * sizeof(double);   // ssim_small_kernel
        fwd = fwd > b ? fwd : b;
    }
    const VifDims vd = vif_dims(H, W);
    for (int s = 0; s < 4; ++s) { const size_t b = fwd_ws_bytes(kVifWin[s], N, vd.h[s], vd.w[s]); fwd = fwd > b ? fwd : b; }
    const size_t pm = msssim_pyr_floats(N, H, W), pv = vif_pyr_floats(N, H, W);
    const size_t pyr = pm > pv ? pm : pv;
    return al256((size_t)(N + 1) * 4) + al256(partial * 8) + 2 * al256(fwd) + al256(hist_extra_words(N) * 4) +
           al256((size_t)N * kRawPerPair * 8) + al256(pyr * 4) + al256(pv * 4) + al256((size_t)N * MMIF_HIST_WORDS * 4) + 256;
}

int carve_metric_ws(MetricWs* w, void* ws, size_t ws_bytes, int N, int H, int W) {
    const size_t need = metric_ws_bytes(N, H, W);
    if (!ws || need == 0 || ws_bytes < need) { set_error("metric workspace too small: %zu < %zu", ws_bytes, need); return MMIF_E_WORKSPACE; }
    if (((uintptr_t)ws) & 255) { set_error("metric workspace must be 256-byte aligned"); return MMIF_E_ALIGN; }
    unsigned char* p = (unsigned char*)ws;
    size_t partial = (size_t)N * ceil_div(H, stats_rows_per_block(N, H)) * 14;
    const size_t pq = (size_t)N * ceil_div(W, 128) * ceil_div(H, kPixelMinRows) * 19;
    const size_t ps = (size_t)N * (((size_t)H * W + 255) / 256) * 8;
    partial = partial > pq ? partial : pq;
    partial = partial > ps ? partial : ps;
    size_t fwd = 0;
    const LevelDims md = msssim_dims(H, W, 11);
    for (int l = 0; l < 5; ++l) {
        size_t b = fwd_ws_bytes(11, N, md.h[l], md.w[l]);
        if (md.k[l] < 11) b = ws_counters_bytes(N) + (size_t)N * (((size_t)md.h[l] * md.w[l] + 255) / 256) * 8 * sizeof(double);   // ssim_small_kernel
        fwd = fwd > b ? fwd : b;
    }
    const VifDims vd = vif_dims(H, W);
    for (int s = 0; s < 4; ++s) { const size_t b = fwd_ws_bytes(kVifWin[s], N, vd.h[s], vd.w[s]); fwd = fwd > b ? fwd : b; }
    const size_t pm = msssim_pyr_floats(N, H, W), pv = vif_pyr_floats(N, H, W);
    w->counters = (unsigned*)p; p += al256((size_t)(N + 1) * 4);
    w->partial = (double*)p; p += al256(partial * 8);
    w->fwd_ws = p; w->fwd_ws_bytes = al256(fwd); p += al256(fwd);
    w->hist_extra = (uint32_t*)p; p += al256(hist_extra_words(N) * 4);
    w->raw = (double*)p; p += al256((size_t)N * kRawPerPair * 8);
    w->pyr = (float*)p; w->pyr_floats = pm > pv ? pm : pv; p += al256(w->pyr_floats * 4);
    w->counts = (uint32_t*)p; p += al256((size_t)N * MMIF_HIST_WORDS * 4);
    w->fwd_ws_b = p; p += al256(fwd);
    w->pyr_b = (float*)p;
    return MMIF_OK;
}

static int run_msssim(const float* a, const float* b, const float* f, int N, int H, int W, int win, float data_range,
                      double* raw /* 5x8 per pair at stride */, long long stride, MetricWs& ws, cudaStream_t st) {
    const LevelDims d = msssim_dims(H, W, win);
    const float* ca = a; const float* cb = b; const float* cf = f;
    float* base = ws.pyr;
    for (int l = 0; l < 5; ++l) {
        int rc = run_ssim_level(ca, cb, cf, N, d.h[l], d.w[l], win, data_range, raw + l * 8, stride, ws, st);
        if (rc) return rc;
        if (l == 4) break;
        const int ho = d.h[l + 1], wo = d.w[l + 1];
        if (d.h[l] < 2 || d.w[l] < 2) { set_error("msssim: level %d is %dx%d, cannot be halved", l, d.h[l], d.w[l]); return MMIF_E_SHAPE; }
        Ptr3 p;
        const size_t per = (size_t)N * ho * wo;
        p.src[0] = ca; p.src[1] = cb; p.src[2] = cf;
        p.dst[0] = base; p.dst[1] = base + per; p.dst[2] = base + 2 * per;
        { const int rc2 = launch_halve(p, N, d.h[l], d.w[l], ho, wo, st); if (rc2) return rc2; }
        ca = p.dst[0]; cb = p.dst[1]; cf = p.dst[2];
        base += 3 * per;
    }
    return MMIF_OK;
}

static int run_vif(const float* a, const float* b, const float* f, int N, int H, int W, double* raw /* 4x8 per pair */,
                   long long stride, MetricWs& ws, cudaStream_t st) {
    const VifDims d = vif_dims(H, W);
    if (!d.ok) { set_error("viff: image %dx%d too small for the 4-scale pyramid (windows 17/9/5/3)", H, W); return MMIF_E_SHAPE; }
    const float* ca = a; const float* cb = b; const float* cf = f;
    float* base = ws.pyr;
    for (int s = 0; s < 4; ++s) {
        const int k = kVifWin[s];
        if (s > 0) {
            Taps taps;
            make_taps(&taps, k, (double)k / 5.0);
            const int ho = d.h[s], wo = d.w[s];
            Ptr3 p;
            const size_t per = (size_t)N * ho * wo;
            p.src[0] = ca; p.src[1] = cb; p.src[2] = cf;
            p.dst[0] = base; p.dst[1] = base + per; p.dst[2] = base + 2 * per;
            int rc = MMIF_OK;
            if (k == 9) rc = launch_bd<9>(p, N, d.h[s - 1], d.w[s - 1], ho, wo, taps, st);
            else if (k == 5) rc = launch_bd<5>(p, N, d.h[s - 1], d.w[s - 1], ho, wo, taps, st);
            else rc = launch_bd<3>(p, N, d.h[s - 1], d.w[s - 1], ho, wo, taps, st);
            if (rc) return rc;
            ca = p.dst[0]; cb = p.dst[1]; cf = p.dst[2];
            base += 3 * per;
        }
        FwdLaunch L;
        memset(&L, 0, sizeof(L));
        L.win = k; L.sigma = (double)k / 5.0; L.epi = EPI_VIF; L.finalize = FIN_SUMS; L.data_range = 255.f;
        L.cfg.pixel_norm = L.cfg.grad_norm = MMIF_NORM_L1;
        // Experiment switch (DESIGN.md section 2): exact central moments instead of the emulation of the reference's fp32
        // window (sum 1 + eps).  Measured: WITHOUT the emulation 26 parity cases fail (random 8-bit images by 5e-5..1e-4),
        // with it only flat-region-dominated real images remain ill-conditioned — so the emulation stays on.
        static const char* vif_plain = getenv("MMIF_VIF_PLAIN_MOMENTS");
        L.plain_moments = (vif_plain && atoi(vif_plain) == 1) ? 1 : 0;
        int rc = launch_moment_fwd(L, ca, cb, cf, N, d.h[s], d.w[s], raw + s * 8, stride, nullptr, ws.fwd_ws, ws.fwd_ws_bytes, st);
        if (rc) return rc;
    }
    return MMIF_OK;
}

static int check_imgs(const void* a, const void* b, const void* f, int N, int H, int W) {
    if (!a || !b || !f) { set_error("null image pointer"); return MMIF_E_NULL; }
    if (N < 1 || H < 1 || W < 1) { set_error("bad shape (%d,%d,%d)", N, H, W); return MMIF_E_SHAPE; }
    if (((uintptr_t)a | (uintptr_t)b | (uintptr_t)f) & 3) { set_error("image pointers must be 4-byte aligned"); return MMIF_E_ALIGN; }
    return MMIF_OK;
}

}  // namespace mmif

using namespace mmif;

extern "C" size_t mmif_metric_workspace_bytes(int N, int H, int W) { return metric_ws_bytes(N, H, W); }

extern "C" int mmif_stats(const float* a, const float* b, const float* f, int N, int H, int W, double* out, void* ws,
                          size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    return launch_stats(a, b, f, N, H, W, out, MMIF_ST_COUNT, w, (cudaStream_t)stream);
}

extern "C" int mmif_stats_bwd(const float* a, const float* b, const float* f, int N, int H, int W, const double* row,
                              const float* gout, float* da, float* db, float* df, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!row || !gout) { set_error("null row or gout"); return MMIF_E_NULL; }
    if ((((uintptr_t)row) & 7) || ((((uintptr_t)gout) | ((uintptr_t)da) | ((uintptr_t)db) | ((uintptr_t)df)) & 3)) {
        set_error("row must be 8-byte, gout and the gradients 4-byte aligned");
        return MMIF_E_ALIGN;
    }
    return launch_stats_bwd(a, b, f, N, H, W, row, gout, da, db, df, (cudaStream_t)stream);
}

extern "C" int mmif_hist(const float* a, const float* b, const float* f, int N, int H, int W, uint32_t* counts, double* ent,
                         void* ws, size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!counts) { set_error("null counts"); return MMIF_E_NULL; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    MMIF_CUDA(cudaMemsetAsync(counts, 0, (size_t)N * MMIF_HIST_WORDS * 4, (cudaStream_t)stream));
    return launch_hist(a, b, f, N, H, W, counts, ent, MMIF_EN_COUNT, w, (cudaStream_t)stream);
}

extern "C" int mmif_qabf(const float* a, const float* b, const float* f, int N, int H, int W, float L, double* out, void* ws,
                         size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    return launch_qabf(a, b, f, N, H, W, L, out, 4, w, (cudaStream_t)stream);
}

/* mmif_qabf plus the five raw sums it is made of (per pair 9 doubles). */
extern "C" int mmif_qabf_raw(const float* a, const float* b, const float* f, int N, int H, int W, float L, double* out, void* ws,
                         size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    return launch_qabf(a, b, f, N, H, W, L, out, MMIF_QABF_RAW_DOUBLES, w, (cudaStream_t)stream, 1);
}

extern "C" int mmif_ssim(const float* a, const float* b, const float* f, int N, int H, int W, int win_size, float data_range,
                         int use_padding, double* out, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    if (use_padding) { set_error("use_padding=True is not built yet"); return MMIF_E_MODE; }
    if (win_size < 1 || win_size > 11) { set_error("ssim window %d unsupported (1..11)", win_size); return MMIF_E_MODE; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = run_ssim_level(a, b, f, N, H, W, win_size, data_range, w.raw + RAW_SSIM, kRawPerPair, w, st); if (rc) return rc;
    const int k = win_size < H ? (win_size < W ? win_size : W) : (H < W ? H : W);
    ssim_out_kernel<<<ceil_div(N, 128), 128, 0, st>>>(w.raw + RAW_SSIM, kRawPerPair, N, 1.0 / ((double)(H - k + 1) * (W - k + 1)), out);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

extern "C" int mmif_msssim(const float* a, const float* b, const float* f, int N, int H, int W, int win_size, float data_range,
                           double* out, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    if (win_size != 11) { set_error("msssim: only the 11-tap window is built"); return MMIF_E_MODE; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = run_msssim(a, b, f, N, H, W, win_size, data_range, w.raw + RAW_MS, kRawPerPair, w, st); if (rc) return rc;
    msssim_out_kernel<<<ceil_div(N, 128), 128, 0, st>>>(w.raw + RAW_MS, kRawPerPair, N, msssim_dims(H, W, win_size), out);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

extern "C" int mmif_viff(const float* a, const float* b, const float* f, int N, int H, int W, double* out, void* ws,
                         size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    rc = run_vif(a, b, f, N, H, W, w.raw + RAW_VIF, kRawPerPair, w, st); if (rc) return rc;
    viff_out_kernel<<<ceil_div(N, 128), 128, 0, st>>>(w.raw + RAW_VIF, kRawPerPair, N, out);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// The four metric families of the suite are independent until the last (tiny) compose kernel: they are
// forked onto three library-owned streams and joined back with events (no host synchronisation; legal
// under stream capture), so the histogram kernel (one 1024-thread CTA per joint, i.e. 2N of the 148 SMs)
// and the small pyramid levels overlap with the bandwidth- / FMA-bound kernels of the other families.
struct SuiteFork { cudaStream_t s[3]; cudaEvent_t fork, join[3]; int dev; bool ok; };
static SuiteFork* suite_fork() {
    static thread_local SuiteFork tab[8];
    static const bool serial = getenv("MMIF_SERIAL") != nullptr;
    if (serial) return nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    SuiteFork* f = nullptr;
    for (int i = 0; i < 8 && !f; ++i) {
        if (tab[i].ok && tab[i].dev == dev) f = &tab[i];
        else if (!tab[i].ok) {
            SuiteFork& t = tab[i];
            bool good = cudaEventCreateWithFlags(&t.fork, cudaEventDisableTiming) == cudaSuccess;
            for (int k = 0; k < 3 && good; ++k)
                good = cudaStreamCreateWithFlags(&t.s[k], cudaStreamNonBlocking) == cudaSuccess &&
                       cudaEventCreateWithFlags(&t.join[k], cudaEventDisableTiming) == cudaSuccess;
            if (!good) { (void)cudaGetLastError(); return nullptr; }
            t.dev = dev; t.ok = true; f = &t;
        }
    }
    return f;
}

extern "C" int mmif_eval_suite(const float* a, const float* b, const float* f, int N, int H, int W, double* out, void* ws,
                               size_t ws_bytes, void* stream) {
    int rc = check_imgs(a, b, f, N, H, W); if (rc) return rc;
    if (!out) { set_error("null out"); return MMIF_E_NULL; }
    if (H < 11 || W < 11) { set_error("eval suite needs H,W >= 11"); return MMIF_E_SHAPE; }
    MetricWs w; rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    SuiteFork* fk = suite_fork();
    cudaStream_t s_ms = st, s_px = st, s_hi = st;
    if (fk) {
        s_ms = fk->s[0]; s_px = fk->s[1]; s_hi = fk->s[2];
        MMIF_CUDA(cudaEventRecord(fk->fork, st));
        for (int k = 0; k < 3; ++k) MMIF_CUDA(cudaStreamWaitEvent(fk->s[k], fk->fork, 0));
    }
    MetricWs wv = w;                  // VIF chain (longest): caller's stream, its own strip workspace + pyramid
    wv.fwd_ws = w.fwd_ws_b; wv.pyr = w.pyr_b;
    int rc_v = run_vif(a, b, f, N, H, W, w.raw + RAW_VIF, kRawPerPair, wv, st);
    // level 0 of the MS-SSIM pyramid is calc_ssim(.., data_range=255) itself (metric.py:379-384)
    int rc_m = run_msssim(a, b, f, N, H, W, 11, 255.f, w.raw + RAW_MS, kRawPerPair, w, s_ms);
    int rc_p = launch_pixel_metrics(a, b, f, N, H, W, 1.5f, w.raw + RAW_STATS, kRawPerPair, w.raw + RAW_QABF, kRawPerPair, w, s_px);
    int rc_h = MMIF_OK;
    if (cudaMemsetAsync(w.counts, 0, (size_t)N * MMIF_HIST_WORDS * 4, s_hi) != cudaSuccess) rc_h = cuda_fail(cudaGetLastError(), "memset");
    if (!rc_h) rc_h = launch_hist(a, b, f, N, H, W, w.counts, w.raw + RAW_ENT, kRawPerPair, w, s_hi);
    if (fk) {                          // always join, even after a launch error, so the streams stay ordered
        for (int k = 0; k < 3; ++k) {
            MMIF_CUDA(cudaEventRecord(fk->join[k], fk->s[k]));
            MMIF_CUDA(cudaStreamWaitEvent(st, fk->join[k], 0));
        }
    }
    if (rc_v) return rc_v;
    if (rc_m) return rc_m;
    if (rc_p) return rc_p;
    if (rc_h) return rc_h;
    suite_out_kernel<<<ceil_div(N, 128), 128, 0, st>>>(w.raw, N, msssim_dims(H, W, 11), 1.0 / ((double)(H - 10) * (W - 10)), out);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

extern "C" int mmif_eval_suite_host(const float* a_host, const float* b_host, const float* f_host, int N, int H, int W,
                                    double* out_host, float* dev_scratch, double* dev_out, void* ws, size_t ws_bytes,
                                    void* stream) {
    if (!a_host || !b_host || !f_host || !out_host || !dev_scratch || !dev_out) { set_error("null pointer"); return MMIF_E_NULL; }
    if (N < 1 || H < 1 || W < 1) { set_error("bad shape"); return MMIF_E_SHAPE; }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)N * H * W;
    MMIF_CUDA(cudaMemcpyAsync(dev_scratch, a_host, n * 4, cudaMemcpyHostToDevice, st));
    MMIF_CUDA(cudaMemcpyAsync(dev_scratch + n, b_host, n * 4, cudaMemcpyHostToDevice, st));
    MMIF_CUDA(cudaMemcpyAsync(dev_scratch + 2 * n, f_host, n * 4, cudaMemcpyHostToDevice, st));
    int rc = mmif_eval_suite(dev_scratch, dev_scratch + n, dev_scratch + 2 * n, N, H, W, dev_out, ws, ws_bytes, stream);
    if (rc) return rc;
    MMIF_CUDA(cudaMemcpyAsync(out_host, dev_out, (size_t)N * MMIF_EVAL_METRICS * 8, cudaMemcpyDeviceToHost, st));
    MMIF_CUDA(cudaStreamSynchronize(st));
    return MMIF_OK;
}

extern "C" int mmif_widen_u8(const unsigned char* src, size_t n, float* dst, void* stream);

extern "C" int mmif_eval_suite_u8(const unsigned char* a, const unsigned char* b, const unsigned char* f, int N, int H, int W,
                                  double* out, float* dev_scratch, void* ws, size_t ws_bytes, void* stream) {
    if (!a || !b || !f || !dev_scratch) { set_error("null pointer"); return MMIF_E_NULL; }
    if (N < 1 || H < 1 || W < 1) { set_error("bad shape"); return MMIF_E_SHAPE; }
    const size_t n = (size_t)N * H * W;
    int rc = mmif_widen_u8(a, n, dev_scratch, stream); if (rc) return rc;
    rc = mmif_widen_u8(b, n, dev_scratch + n, stream); if (rc) return rc;
    rc = mmif_widen_u8(f, n, dev_scratch + 2 * n, stream); if (rc) return rc;
    return mmif_eval_suite(dev_scratch, dev_scratch + n, dev_scratch + 2 * n, N, H, W, out, ws, ws_bytes, stream);
}

extern "C" int mmif_eval_suite_u8_host(const unsigned char* a_host, const unsigned char* b_host, const unsigned char* f_host, int N,
                                       int H, int W, double* out_host, unsigned char* dev_u8, float* dev_scratch, double* dev_out,
                                       void* ws, size_t ws_bytes, void* stream) {
    if (!a_host || !b_host || !f_host || !out_host || !dev_u8 || !dev_scratch || !dev_out) { set_error("null pointer"); return MMIF_E_NULL; }
    if (N < 1 || H < 1 || W < 1) { set_error("bad shape"); return MMIF_E_SHAPE; }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)N * H * W;
    const size_t n16 = (n + 15) / 16 * 16;                       // keep the three device images 16-byte aligned
    MMIF_CUDA(cudaMemcpyAsync(dev_u8, a_host, n, cudaMemcpyHostToDevice, st));
    MMIF_CUDA(cudaMemcpyAsync(dev_u8 + n16, b_host, n, cudaMemcpyHostToDevice, st));
    MMIF_CUDA(cudaMemcpyAsync(dev_u8 + 2 * n16, f_host, n, cudaMemcpyHostToDevice, st));
    int rc = mmif_eval_suite_u8(dev_u8, dev_u8 + n16, dev_u8 + 2 * n16, N, H, W, dev_out, dev_scratch, ws, ws_bytes, stream);
    if (rc) return rc;
    MMIF_CUDA(cudaMemcpyAsync(out_host, dev_out, (size_t)N * MMIF_EVAL_METRICS * 8, cudaMemcpyDeviceToHost, st));
    MMIF_CUDA(cudaStreamSynchronize(st));
    return MMIF_OK;
}

extern "C" int mmif_tv_loss(const float* x, int N, int H, int W, int norm, float weight, double* out, void* ws, size_t ws_bytes,
                            void* stream) {
    if (!x || !out) { set_error("null pointer"); return MMIF_E_NULL; }
    if (norm != MMIF_NORM_L1 && norm != MMIF_NORM_L2) { set_error("unsupported norm"); return MMIF_E_MODE; }
    MetricWs w; int rc = carve_metric_ws(&w, ws, ws_bytes, N, H, W); if (rc) return rc;
    return launch_tv(x, N, H, W, norm, weight, out, w, (cudaStream_t)stream);
}
