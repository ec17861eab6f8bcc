// Per-pixel metric families of reference core/metric.py: first/second-order statistics
// (SD/AG/SF/MSE/CC/SCD), histograms + entropies (EN/CE/MI), edge preservation (Qabf/Nabf/Labf),
// and TVLoss of core/loss.py.  Every kernel reads its inputs once, accumulates in registers,
// reduces per block with warp shuffles in double, and the last block of a pair finishes that pair
// in a fixed order (deterministic, no float atomics).
#include <stdlib.h>
#include "metrics.cuh"

namespace mmif {

// =============================================================================== statistics + Qabf
// One pass over (a, b, f) serves both per-pixel families: the first/second-order statistics
// (SD/AG/SF/MSE/CC/SCD, metric.py:25-99) are bandwidth-only work and ride for free under the
// transcendental-bound edge-preservation sums (Qabf/Nabf/Labf, metric.py:192-286).
// thread = column, marching down a chunk of rows with a 3-row sliding window (reflect borders);
// one coalesced load per image per row, the left / right neighbours come from warp shuffles (the two
// edge lanes of a warp fetch theirs), every statistic lives in registers.
// sums: 0 Sa 1 Sb 2 Sf 3 Saa 4 Sbb 5 Sff 6 Sab 7 Saf 8 Sbf 9 Sag 10 Sdx2 11 Sdy2 12 S(a-f)^2 13 S(b-f)^2
//       then (Qabf) Sq, Sw, Sn (modified), Sl, Sn_unmodified
constexpr int kStatK = 14;
constexpr int kQK = 5;

__device__ __forceinline__ float sqrt_fast(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rcp_fast(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float ex2_fast(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// atan2(y, x) in (-pi, pi]: |error| < 1.5e-7 (degree-8 minimax in (min/max)^2, fp32 Horner); atan2(+0, +0) = 0,
// atan2(+0, x < 0) = pi like the reference's torch.atan2 (the Sobel differences of a flat patch are +0).
__device__ __forceinline__ float atan2_fast(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float a = (mx > 0.f) ? mn * rcp_fast(mx) : 0.f;       // 1-ulp reciprocal: |d atan| <= 1.2e-7
    const float s = a * a;
    float p = 0.002456702059134841f;
    p = fmaf(p, s, -0.014401260763406754f);
    p = fmaf(p, s, 0.03978104889392853f);
    p = fmaf(p, s, -0.07234840840101242f);
    p = fmaf(p, s, 0.10498937219381332f);
    p = fmaf(p, s, -0.14161226153373718f);
    p = fmaf(p, s, 0.19985906779766083f);
    p = fmaf(p, s, -0.33332598209381104f);
    p = fmaf(p, s, 0.9999998807907104f);
    float r = p * a;
    if (ay > ax) r = 1.5707963267948966f - r;
    if (x < 0.f) r = 3.141592653589793f - r;
    return copysignf(r, y);
}
// gamma / (1 + exp(-k (v - sigma)))   (metric.py:224-225)
__device__ __forceinline__ float sigmoid_q(float gamma, float k, float sigma, float v) {
    const float e = ex2_fast(-k * 1.4426950408889634f * (v - sigma));
    return gamma * rcp_fast(1.f + e);
}

template <bool STATS, bool QABF>
__global__ void __launch_bounds__(128)
pixel_metrics_kernel(const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ F, int H, int W, int rpb,
                     float Lexp, double* partial, unsigned* counters, double* out_s, long long sstride, double* out_q,
                     long long qstride, int q_raw) {
    constexpr int K = (STATS ? kStatK : 0) + (QABF ? kQK : 0);
    constexpr int QO = STATS ? kStatK : 0;
    __shared__ double red[K * 4];
    __shared__ int flag;
    const int n = blockIdx.z;
    const int blk = blockIdx.y * gridDim.x + blockIdx.x, nblk = gridDim.x * gridDim.y;
    const size_t off = (size_t)n * H * W;
    const float* img[3] = {A + off, Bm + off, F + off};
    const int c_raw = blockIdx.x * 128 + threadIdx.x;
    const bool colok = c_raw < W;
    const int c = min(c_raw, W - 1);
    const int lane = threadIdx.x & 31;
    const bool edgeL = (c == 0), edgeR = (c == W - 1);
    const bool ldL = (lane == 0) && !edgeL, ldR = (lane == 31) && !edgeR;
    const int r0 = blockIdx.y * rpb, r1 = min(r0 + rpb, H);
    float s[K];
#pragma unroll
    for (int i = 0; i < K; ++i) s[i] = 0.f;
    float dA[3], dB[3], sA[3], sB[3], pc[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) dA[k] = dB[k] = sA[k] = sB[k] = pc[k] = 0.f;
    float pfr = 0.f;
    // the loads of row r+1 are issued before row r is consumed (one row of prefetch hides the global latency)
    float nuc[3], nxl[3], nxr[3];
    auto fetch = [&](int r) {
        const int rr = (r < 0) ? -r : ((r >= H) ? 2 * H - 2 - r : r);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float* row = img[k] + (size_t)rr * W + c;
            nuc[k] = __ldg(row);
            nxl[k] = ldL ? __ldg(row - 1) : 0.f;
            nxr[k] = ldR ? __ldg(row + 1) : 0.f;
        }
    };
    fetch(r0 - 1);
    for (int r = r0 - 1; r <= r1; ++r) {
        float gx[3], gy[3], uc[3], xls[3], xrs[3], upf = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) { uc[k] = nuc[k]; xls[k] = nxl[k]; xrs[k] = nxr[k]; }
        if (r < r1) fetch(r + 1);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float xl = xls[k], xr = xrs[k];
            float um = __shfl_up_sync(0xffffffffu, uc[k], 1), up = __shfl_down_sync(0xffffffffu, uc[k], 1);
            if (lane == 0) um = xl;
            if (lane == 31) up = xr;
            if (edgeL) um = up;                              // reflect: column -1 is column 1
            if (edgeR) up = um;                              //          column W is column W-2
            if (k == 2) upf = up;
            if (QABF) {
                const float d = up - um, sm = um + 2.f * uc[k] + up;
                gx[k] = dA[k] + 2.f * dB[k] + d;
                gy[k] = sm - sA[k];
                dA[k] = dB[k]; dB[k] = d; sA[k] = sB[k]; sB[k] = sm;
            }
        }
        if (r >= r0 + 1 && colok) {            // everything below describes pixel row r-1
            if (STATS) {
                const float fa = pc[0], fb = pc[1], ff = pc[2];
                const bool hasx = !edgeR, hasy = (r < H);
                s[0] += fa; s[1] += fb; s[2] += ff;
                s[3] = fmaf(fa, fa, s[3]); s[4] = fmaf(fb, fb, s[4]); s[5] = fmaf(ff, ff, s[5]);
                s[6] = fmaf(fa, fb, s[6]); s[7] = fmaf(fa, ff, s[7]); s[8] = fmaf(fb, ff, s[8]);
                const float dx = pfr - ff, dy = uc[2] - ff;
                if (hasx) s[10] = fmaf(dx, dx, s[10]);
                if (hasy) s[11] = fmaf(dy, dy, s[11]);
                if (hasx && hasy) s[9] += sqrt_fast((dx * dx + dy * dy) * 0.5f);  // metric.py:44
                const float ea = fa - ff, eb = fb - ff;
                s[12] = fmaf(ea, ea, s[12]); s[13] = fmaf(eb, eb, s[13]);
            }
            if (QABF) {
                float g[3], al[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) { g[k] = sqrt_fast(fmaf(gx[k], gx[k], gy[k] * gy[k])); al[k] = atan2_fast(gy[k], gx[k]); }
                float Q[2], w[2];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const float mx = fmaxf(g[k], g[2]), mn = fminf(g[k], g[2]);
                    const float G = (mx > 0.f) ? mn * rcp_fast(mx) : 0.f;                // 0/0 -> 0, metric.py:213-215
                    const float Aa = fabsf(fabsf(al[k] - al[2]) - 1.5707963267948966f) * 0.6366197723675814f;
                    Q[k] = sigmoid_q(0.9994f, 15.f, 0.5f, G) * sigmoid_q(0.9879f, 22.f, 0.8f, Aa);   // metric.py:218-225
                    w[k] = (Lexp == 1.5f) ? g[k] * sqrt_fast(g[k]) : powf(g[k], Lexp);     // eval.py:45 uses L=1.5
                }
                const float gmax = fmaxf(g[0], g[1]);
                const float lossw = (1.f - Q[0]) * w[0] + (1.f - Q[1]) * w[1];
                s[QO + 0] += Q[0] * w[0] + Q[1] * w[1];
                s[QO + 1] += w[0] + w[1];
                if (g[2] > gmax) { s[QO + 2] += lossw; s[QO + 4] += (2.f - Q[0] - Q[1]) * (w[0] + w[1]); }
                if (g[2] <= gmax) s[QO + 3] += lossw;
            }
        }
        pc[0] = uc[0]; pc[1] = uc[1]; pc[2] = uc[2]; pfr = upf;
    }
    double acc[K];
#pragma unroll
    for (int i = 0; i < K; ++i) acc[i] = (double)s[i];
    double t[K];
    if (!block_finish<K, 128>(acc, red, &flag, partial, counters, n, blk, nblk, t)) return;
    // ---- last block, thread 0: the metrics of this pair (double arithmetic on the raw sums) ----
    if (STATS) {
        const double P = (double)H * (double)W;
        const double ma = t[0] / P, mb = t[1] / P, mf = t[2] / P;
        const double vaa = t[3] - t[0] * t[0] / P, vbb = t[4] - t[1] * t[1] / P, vff = t[5] - t[2] * t[2] / P;   // P * variance
        const double cab = t[6] - t[0] * t[1] / P, caf = t[7] - t[0] * t[2] / P, cbf = t[8] - t[1] * t[2] / P;   // P * covariance
        double* o = out_s + (size_t)n * sstride;
        o[MMIF_ST_MEAN_F] = mf;
        o[MMIF_ST_SD] = sqrt(fmax(vff, 0.0) / P);
        o[MMIF_ST_AG] = t[9] / ((double)(H - 1) * (double)(W - 1));
        o[MMIF_ST_SF] = sqrt(t[11] / ((double)(H - 1) * (double)W) + t[10] / ((double)H * (double)(W - 1)));
        o[MMIF_ST_MSE_AF] = t[12] / (255.0 * 255.0) / P;                       // metric.py:63-68
        o[MMIF_ST_MSE_BF] = t[13] / (255.0 * 255.0) / P;
        o[MMIF_ST_CC_AF] = caf / sqrt(vaa * vff);                              // metric.py:80-91
        o[MMIF_ST_CC_BF] = cbf / sqrt(vbb * vff);
        // scd = cc(f-a, b) + cc(f-b, a) (metric.py:95-99) from second moments
        const double v_fa = vff + vaa - 2.0 * caf, v_fb = vff + vbb - 2.0 * cbf;
        o[MMIF_ST_SCD] = (cbf - cab) / sqrt(v_fa * vbb) + (caf - cab) / sqrt(v_fb * vaa);
        o[MMIF_ST_MEAN_A] = ma; o[MMIF_ST_MEAN_B] = mb;
        o[MMIF_ST_SD_A] = sqrt(fmax(vaa, 0.0) / P); o[MMIF_ST_SD_B] = sqrt(fmax(vbb, 0.0) / P);
        o[MMIF_ST_CC_AB] = cab / sqrt(vaa * vbb);
        o[14] = 0.0; o[15] = 0.0;
    }
    if (QABF) {
        double* o = out_q + (size_t)n * qstride;
        o[0] = t[QO + 0] / t[QO + 1]; o[1] = t[QO + 2] / t[QO + 1]; o[2] = t[QO + 3] / t[QO + 1]; o[3] = t[QO + 4] / t[QO + 1];
        if (q_raw) {                     // the five raw sums as well: a batch is combined as sum / sum (metric.py:233-256 with N > 1)
#pragma unroll
            for (int i = 0; i < kQK; ++i) o[4 + i] = t[QO + i];
        }
    }
}

int pixel_rows_per_block(int N, int H, int W) {
    int rpb = 32;
    while (rpb > kPixelMinRows && (long long)N * ceil_div(W, 128) * ceil_div(H, rpb) < 4 * 148) rpb >>= 1;
    return rpb;
}
int stats_rows_per_block(int N, int H) {       // TVLoss
    int rpb = (int)(((long long)N * H + 591) / 592);
    return rpb < 1 ? 1 : (rpb > 32 ? 32 : rpb);
}

int launch_pixel_metrics(const float* a, const float* b, const float* f, int N, int H, int W, float L, double* out_s,
                         long long sstride, double* out_q, long long qstride, MetricWs& ws, cudaStream_t st, int q_raw) {
    if (H < 2 || W < 2) { set_error("stats / qabf: H and W must be >= 2"); return MMIF_E_SHAPE; }
    const int rpb = pixel_rows_per_block(N, H, W);
    dim3 grid(ceil_div(W, 128), ceil_div(H, rpb), N);
    if (out_s && out_q)
        pixel_metrics_kernel<true, true><<<grid, 128, 0, st>>>(a, b, f, H, W, rpb, L, ws.partial, ws.counters, out_s, sstride, out_q, qstride, q_raw);
    else if (out_s)
        pixel_metrics_kernel<true, false><<<grid, 128, 0, st>>>(a, b, f, H, W, rpb, L, ws.partial, ws.counters, out_s, sstride, out_q, qstride, q_raw);
    else
        pixel_metrics_kernel<false, true><<<grid, 128, 0, st>>>(a, b, f, H, W, rpb, L, ws.partial, ws.counters, out_s, sstride, out_q, qstride, q_raw);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
int launch_stats(const float* a, const float* b, const float* f, int N, int H, int W, double* out, long long ostride, MetricWs& ws,
                 cudaStream_t st) {
    return launch_pixel_metrics(a, b, f, N, H, W, 1.5f, out, ostride, nullptr, 0, ws, st);
}
int launch_qabf(const float* a, const float* b, const float* f, int N, int H, int W, float L, double* out, long long ostride,
                MetricWs& ws, cudaStream_t st, int q_raw) {
    return launch_pixel_metrics(a, b, f, N, H, W, L, nullptr, 0, out, ostride, ws, st, q_raw);
}

// =============================================================================== statistics gradient
// Gradient of sum_c gout[c] * stat[c] over the MMIF_ST_* columns of one batch row.  Every statistic except AG and SF is
// a function of the batch means and (co)variances of (a, b, f), so its gradient w.r.t. an image x is affine in the
// centred pixels: dx = c0[x] + K[x][a] (a - ma) + K[x][b] (b - mb) + K[x][f] (f - mf).  dC_xy / dx_i = (y_i - my) / P:
// the mean terms cancel.  AG and SF add their forward-difference stencil terms to df.  Coefficients are formed once
// per block in double; a zero sd or a 0/0 correlation makes its coefficients NaN, so NaN reaches every pixel, as the
// reference's pow(0.5) at 0 and 0/0 correlations do under autograd.  A column whose gout is exactly 0 is skipped.
struct StatsBwdCoef {
    double c0[3], K[3][3], mu[3];
    double kag, ksv, ksh;        // AG per-stencil factor, SF vertical / horizontal factors
};

// d/dx, d/dy of g * corr(x, y) (metric.py:80-91) with sx, sy the population sds and r the correlation.
__device__ void cc_coef(StatsBwdCoef& c, int x, int y, double sx, double sy, double r, double g, double P) {
    if (sx == 0.0 || sy == 0.0) {
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        c.K[x][x] += nan; c.K[x][y] += nan; c.K[y][x] += nan; c.K[y][y] += nan;
        return;
    }
    const double m = g / (P * sx * sy);
    c.K[x][y] += m; c.K[y][x] += m;
    c.K[x][x] -= g * r / (P * sx * sx);
    c.K[y][y] -= g * r / (P * sy * sy);
}

// d/d(src, other, f) of g * corr(f - src, other): one term of scd (metric.py:95-99).
__device__ void scd_coef(StatsBwdCoef& c, int s, int o, double Css, double Coo, double Cff, double Csf, double Cof, double Cso,
                         double g, double P) {
    const double su = sqrt(fmax(Cff + Css - 2.0 * Csf, 0.0)), so = sqrt(Coo);
    if (su == 0.0 || so == 0.0) {
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        for (int x = 0; x < 3; ++x) for (int y = 0; y < 3; ++y) c.K[x][y] += nan;
        return;
    }
    const double r = (Cof - Cso) / (su * so);
    const double A = g / (P * su * so), B = g * r / (P * su * su), C = g * r / (P * so * so);
    // u = f - src, v = other:  gu = A (v - mv) - B (u - mu),  gv = A (u - mu) - C (v - mv);  df += gu, dsrc -= gu, dother += gv
    c.K[2][o] += A; c.K[2][2] -= B; c.K[2][s] += B;
    c.K[s][o] -= A; c.K[s][2] += B; c.K[s][s] -= B;
    c.K[o][2] += A; c.K[o][s] -= A; c.K[o][o] -= C;
}

__device__ void stats_bwd_coef(StatsBwdCoef& c, const double* row, const float* gout, int N, int H, int W) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    const double P = (double)N * H * W;
    const double ma = row[MMIF_ST_MEAN_A], mb = row[MMIF_ST_MEAN_B], mf = row[MMIF_ST_MEAN_F];
    const double sa = row[MMIF_ST_SD_A], sb = row[MMIF_ST_SD_B], sf = row[MMIF_ST_SD];
    // covariances from the correlations; a constant image has zero covariance with anything
    const double Caf = (sa == 0.0 || sf == 0.0) ? 0.0 : row[MMIF_ST_CC_AF] * sa * sf;
    const double Cbf = (sb == 0.0 || sf == 0.0) ? 0.0 : row[MMIF_ST_CC_BF] * sb * sf;
    const double Cab = (sa == 0.0 || sb == 0.0) ? 0.0 : row[MMIF_ST_CC_AB] * sa * sb;
    for (int x = 0; x < 3; ++x) { c.c0[x] = 0.0; for (int y = 0; y < 3; ++y) c.K[x][y] = 0.0; }
    c.mu[0] = ma; c.mu[1] = mb; c.mu[2] = mf;
    c.kag = c.ksv = c.ksh = 0.0;
    double g[MMIF_ST_COUNT];
    for (int i = 0; i < MMIF_ST_COUNT; ++i) g[i] = (double)gout[i];
    if (g[MMIF_ST_MEAN_F] != 0.0) c.c0[2] += g[MMIF_ST_MEAN_F] / P;
    if (g[MMIF_ST_SD] != 0.0) c.K[2][2] += (sf == 0.0) ? nan : g[MMIF_ST_SD] / (P * sf);
    if (g[MMIF_ST_AG] != 0.0) c.kag = g[MMIF_ST_AG] / ((double)N * (H - 1) * (W - 1));
    if (g[MMIF_ST_SF] != 0.0) {
        const double v = row[MMIF_ST_SF];
        c.ksv = (v == 0.0) ? nan : g[MMIF_ST_SF] / (v * ((double)N * (H - 1) * W));
        c.ksh = (v == 0.0) ? nan : g[MMIF_ST_SF] / (v * ((double)N * H * (W - 1)));
    }
    for (int s = 0; s < 2; ++s) {                       // mse(src, f) = E[(src - f)^2] / 255^2 (metric.py:63-68)
        const double gm = g[MMIF_ST_MSE_AF + s];
        if (gm == 0.0) continue;
        const double m = 2.0 * gm / (255.0 * 255.0 * P), d = m * (c.mu[s] - mf);
        c.c0[s] += d; c.c0[2] -= d;
        c.K[s][s] += m; c.K[s][2] -= m; c.K[2][s] -= m; c.K[2][2] += m;
    }
    if (g[MMIF_ST_CC_AF] != 0.0) cc_coef(c, 0, 2, sa, sf, row[MMIF_ST_CC_AF], g[MMIF_ST_CC_AF], P);
    if (g[MMIF_ST_CC_BF] != 0.0) cc_coef(c, 1, 2, sb, sf, row[MMIF_ST_CC_BF], g[MMIF_ST_CC_BF], P);
    if (g[MMIF_ST_CC_AB] != 0.0) cc_coef(c, 0, 1, sa, sb, row[MMIF_ST_CC_AB], g[MMIF_ST_CC_AB], P);
    if (g[MMIF_ST_MEAN_A] != 0.0) c.c0[0] += g[MMIF_ST_MEAN_A] / P;
    if (g[MMIF_ST_MEAN_B] != 0.0) c.c0[1] += g[MMIF_ST_MEAN_B] / P;
    if (g[MMIF_ST_SD_A] != 0.0) c.K[0][0] += (sa == 0.0) ? nan : g[MMIF_ST_SD_A] / (P * sa);
    if (g[MMIF_ST_SD_B] != 0.0) c.K[1][1] += (sb == 0.0) ? nan : g[MMIF_ST_SD_B] / (P * sb);
    if (g[MMIF_ST_SCD] != 0.0) {                        // scd = cc(f - a, b) + cc(f - b, a)
        scd_coef(c, 0, 1, sa * sa, sb * sb, sf * sf, Caf, Cbf, Cab, g[MMIF_ST_SCD], P);
        scd_coef(c, 1, 0, sb * sb, sa * sa, sf * sf, Cbf, Caf, Cab, g[MMIF_ST_SCD], P);
    }
}

// 0.5 / sqrt(0.5 (dx^2 + dy^2)) of one AG stencil (metric.py:44) in IEEE float32: a stencil with dx = dy = 0 gives inf,
// so its dx * w and dy * w are 0 * inf = NaN on exactly its three pixels, as the reference's autograd gives.
__device__ __forceinline__ float ag_w(float dx, float dy) {
    const float q = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    return __fdiv_rn(0.5f, __fsqrt_rn(__fmul_rn(q, 0.5f)));
}

constexpr int kSbRows = 4;     // consecutive rows per thread: a 32 x 8 block covers a tile of 32 x 32 pixels
constexpr int kSbBlocksPerSM = 3;

// Gather form: the thread of pixel (i, j) writes its three outputs once, reading its own pixel, its neighbours and the
// AG stencils (i, j), (i, j-1), (i-1, j) it belongs to.  No atomics: the result is deterministic.  A block forms the
// coefficients once and then strides over the 32 x 32 tiles of the batch.
__global__ void __launch_bounds__(256, kSbBlocksPerSM)
stats_bwd_kernel(const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ F, int N, int H, int W,
                 const double* __restrict__ row, const float* __restrict__ gout, float* da, float* db, float* df) {
    __shared__ StatsBwdCoef cs;
    if (threadIdx.x == 0 && threadIdx.y == 0) stats_bwd_coef(cs, row, gout, N, H, W);
    __syncthreads();
    const StatsBwdCoef& c = cs;
    const bool stencil = df && (c.kag != 0.0 || c.ksv != 0.0 || c.ksh != 0.0);
    const int tx = (W + 31) / 32, ty = (H + 8 * kSbRows - 1) / (8 * kSbRows);
    const long long ntiles = (long long)tx * ty * N;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int j = (int)(tile % tx) * 32 + threadIdx.x;
        const int i0 = (int)((tile / tx) % ty) * (8 * kSbRows) + threadIdx.y * kSbRows;     // this thread's kSbRows rows
        const size_t off = (size_t)(tile / ((long long)tx * ty)) * H * W;
        if (j >= W || i0 >= H) continue;
        const float *a = A + off, *b = Bm + off, *f = F + off;
        // every load first (clamped addresses, unused values are ignored), so a thread has all of them in flight at once
        const int jl = max(j - 1, 0), jr = min(j + 1, W - 1);
        float va[kSbRows], vb[kSbRows], fc[kSbRows + 2], fl[kSbRows + 2], fr[kSbRows + 2];   // f rows i0-1 .. i0+kSbRows
#pragma unroll
        for (int k = 0; k < kSbRows; ++k) {
            const size_t r = (size_t)min(i0 + k, H - 1) * W;
            va[k] = __ldg(a + r + j); vb[k] = __ldg(b + r + j);
        }
#pragma unroll
        for (int k = 0; k < kSbRows + 2; ++k) {
            const size_t r = (size_t)min(max(i0 - 1 + k, 0), H - 1) * W;
            fc[k] = __ldg(f + r + j);
            fl[k] = stencil ? __ldg(f + r + jl) : 0.f;
            fr[k] = stencil ? __ldg(f + r + jr) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < kSbRows; ++k) {
            const int i = i0 + k;
            if (i >= H) break;
            const size_t q = off + (size_t)i * W + j;
            const float fcc = fc[k + 1];
            const double ca = (double)va[k] - c.mu[0], cb = (double)vb[k] - c.mu[1], cf = (double)fcc - c.mu[2];
            if (da) da[q] = (float)(c.c0[0] + c.K[0][0] * ca + c.K[0][1] * cb + c.K[0][2] * cf);
            if (db) db[q] = (float)(c.c0[1] + c.K[1][0] * ca + c.K[1][1] * cb + c.K[1][2] * cf);
            if (!df) continue;
            double v = c.c0[2] + c.K[2][0] * ca + c.K[2][1] * cb + c.K[2][2] * cf;
            if (stencil) {
                const bool up = i > 0, dn = i + 1 < H, lf = j > 0, rt = j + 1 < W;
                const float fu = fc[k], fd = fc[k + 2], fle = fl[k + 1], fri = fr[k + 1];
                if (c.ksv != 0.0 || c.ksh != 0.0) {          // sf (metric.py:50-59): dv = f(i+1,j) - f(i,j), dh = f(i,j+1) - f(i,j)
                    const double dvu = up ? (double)fcc - fu : 0.0, dvd = dn ? (double)fd - fcc : 0.0;
                    const double dhl = lf ? (double)fcc - fle : 0.0, dhr = rt ? (double)fri - fcc : 0.0;
                    v += c.ksv * (dvu - dvd) + c.ksh * (dhl - dhr);
                }
                if (c.kag != 0.0) {                          // ag (metric.py:38-46) on the (H-1) x (W-1) stencil grid
                    float t = 0.f;
                    if (dn && rt) {                          // stencil (i, j): this pixel is its base
                        const float dx = fri - fcc, dy = fd - fcc, w = ag_w(dx, dy);
                        t = -(dx * w) - (dy * w);
                    }
                    if (dn && lf) {                          // stencil (i, j-1): this pixel is its right neighbour
                        const float dx = fcc - fle, dy = fl[k + 2] - fle;
                        t += dx * ag_w(dx, dy);
                    }
                    if (up && rt) {                          // stencil (i-1, j): this pixel is its lower neighbour
                        const float dx = fr[k] - fu, dy = fcc - fu;
                        t += dy * ag_w(dx, dy);
                    }
                    v += c.kag * (double)t;
                }
            }
            df[q] = (float)v;
        }
    }
}

int launch_stats_bwd(const float* a, const float* b, const float* f, int N, int H, int W, const double* row, const float* gout,
                     float* da, float* db, float* df, cudaStream_t st) {
    if (H < 2 || W < 2) { set_error("stats_bwd: H and W must be >= 2"); return MMIF_E_SHAPE; }
    if (!da && !db && !df) return MMIF_OK;
    const long long tiles = (long long)ceil_div(W, 32) * ceil_div(H, 8 * kSbRows) * N;
    const int grid = (int)(tiles < 148 * kSbBlocksPerSM ? tiles : 148 * kSbBlocksPerSM);
    stats_bwd_kernel<<<grid, dim3(32, 8), 0, st>>>(a, b, f, N, H, W, row, gout, da, db, df);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// =============================================================================== histograms
// Bin rule of torch.histc(im, 256, 0, 256) and np.histogram2d(.., 256, ((0,256),(0,256)))
// (metric.py:113, 141-143): bin = floor(v) for 0 <= v < 256, v == 256 -> 255, -0.0 -> 0,
// anything else (v < 0, v > 256, NaN) is dropped; a joint sample is dropped if either value is.
//
// grid (2*S, N), 1024 threads, one CTA per SM: CTA (joint j, split s) of pair n holds the WHOLE
// 256x256 joint histogram of (source_j, f) in 128 KB of shared memory as packed 15-bit counters
// (two per word, bit 15 / bit 31 = guard): the thread whose increment sets a guard bit clears it and
// moves the 32768 counts to the global histogram, so a pixel costs exactly one shared-memory atomic
// (measured ATOMS rate: 7.6 /clk/SM, independent of the bin count) and is read by two CTAs only.
// The three marginals are row / column sums of the joints (+ the samples whose partner was dropped).
// S == 1 (enough pairs to fill the GPU): the CTA stores its histogram and finishes the entropy family
// of its joint from shared memory — one launch, no finalize kernel.  S > 1 (few pairs): the splits
// add their counts to the global histogram and the last CTA to arrive finishes from there.
constexpr int kHT = 1024;        // threads per histogram CTA
constexpr int kClogN = 4096;     // c * log2(c) table entries (shared memory, built per CTA)
constexpr int kHistExtraWords = 1056;   // per pair: [j][exs 256 | exf 256] + 2 arrival counters + pad

struct HistSmem {
    uint32_t jh[32768];
    double clog[kClogN];
    double red[5 * (kHT / 32)];
    uint32_t exs[256], exf[256], rows[256], cols[256];
    int flag;
};

__device__ __forceinline__ void hist_add(HistSmem& sm, uint32_t* gj, uint32_t idx) {
    const uint32_t delta = 1u << ((idx & 1u) << 4);
    const uint32_t old = atomicAdd(&sm.jh[idx >> 1], delta);
    if (((old + delta) & ~old) & (delta << 15)) {          // this increment set the guard bit of its counter
        atomicSub(&sm.jh[idx >> 1], delta << 15);
        atomicAdd(&gj[idx], 0x8000u);
    }
}
__device__ __forceinline__ void hist_count(HistSmem& sm, uint32_t* gj, float vs, float vf) {
    // fast path: floor(v) + 2^23 by a round-down add; 0 <= v < 256 <=> the biased bits are <= 255
    const uint32_t us = __float_as_uint(__fadd_rd(vs, 8388608.f)) - 0x4B000000u;
    const uint32_t uf = __float_as_uint(__fadd_rd(vf, 8388608.f)) - 0x4B000000u;
    if (max(us, uf) <= 255u) { hist_add(sm, gj, us * 256u + uf); return; }
    // rare: a value of exactly 256 (bin 255) or a sample to drop
    const bool oks = (vs >= 0.f) && (vs <= 256.f), okf = (vf >= 0.f) && (vf <= 256.f);
    const int bs = min(__float2int_rz(vs), 255), bf = min(__float2int_rz(vf), 255);
    if (oks && okf) hist_add(sm, gj, (uint32_t)(bs * 256 + bf));
    else if (oks) atomicAdd(&sm.exs[bs], 1u);                  // source counted in its marginal only
    else if (okf) atomicAdd(&sm.exf[bf], 1u);                  // f counted in its marginal only
}

__global__ void __launch_bounds__(kHT, 1)
hist_kernel(const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ F, long long P, int S,
            uint32_t* counts, uint32_t* extra, double* ent, long long estride) {
    extern __shared__ __align__(16) unsigned char hist_smem_raw[];
    HistSmem& sm = *reinterpret_cast<HistSmem*>(hist_smem_raw);
    const int n = blockIdx.y, j = blockIdx.x & 1, s = blockIdx.x >> 1;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    {
        uint4* z = reinterpret_cast<uint4*>(sm.jh);
        for (int i = t; i < 32768 / 4; i += kHT) z[i] = make_uint4(0u, 0u, 0u, 0u);
        for (int c = t; c < kClogN; c += kHT) sm.clog[c] = c ? (double)c * log2((double)c) : 0.0;
        if (t < 256) { sm.exs[t] = 0u; sm.exf[t] = 0u; sm.rows[t] = 0u; sm.cols[t] = 0u; }
    }
    __syncthreads();
    const float* src = (j == 0 ? A : Bm) + (size_t)n * P;
    const float* f = F + (size_t)n * P;
    uint32_t* cn = counts + (size_t)n * MMIF_HIST_WORDS;
    uint32_t* gj = cn + 768 + (size_t)j * 65536;
    uint32_t* ex = extra + (size_t)n * kHistExtraWords;
    long long p0 = P * s / S, p1 = P * (s + 1) / S;
    const bool vec = ((P & 3) == 0) && ((((uintptr_t)src | (uintptr_t)f) & 15) == 0);
    if (vec) {
        p0 &= ~3ll;
        if (s + 1 < S) p1 &= ~3ll;
        const float4* s4 = reinterpret_cast<const float4*>(src);
        const float4* f4 = reinterpret_cast<const float4*>(f);
        const long long q1 = p1 >> 2;
        long long q = (p0 >> 2) + t;
        for (; q + kHT < q1; q += 2 * kHT) {            // two independent float4 pairs in flight
            const float4 a0 = __ldg(s4 + q), b0 = __ldg(f4 + q), a1 = __ldg(s4 + q + kHT), b1 = __ldg(f4 + q + kHT);
            hist_count(sm, gj, a0.x, b0.x); hist_count(sm, gj, a0.y, b0.y);
            hist_count(sm, gj, a0.z, b0.z); hist_count(sm, gj, a0.w, b0.w);
            hist_count(sm, gj, a1.x, b1.x); hist_count(sm, gj, a1.y, b1.y);
            hist_count(sm, gj, a1.z, b1.z); hist_count(sm, gj, a1.w, b1.w);
        }
        for (; q < q1; q += kHT) {
            const float4 a0 = __ldg(s4 + q), b0 = __ldg(f4 + q);
            hist_count(sm, gj, a0.x, b0.x); hist_count(sm, gj, a0.y, b0.y);
            hist_count(sm, gj, a0.z, b0.z); hist_count(sm, gj, a0.w, b0.w);
        }
    } else {
        for (long long p = p0 + t; p < p1; p += kHT) hist_count(sm, gj, __ldg(src + p), __ldg(f + p));
    }
    __threadfence();
    __syncthreads();
    const bool fused = (S == 1);
    if (!fused) {
        // ---- split mode: add this split to the global histogram; the last split of (n, j) finishes ----
        for (int i = t; i < 32768; i += kHT) {
            const uint32_t w = sm.jh[i];
            if (w & 0xFFFFu) atomicAdd(&gj[2 * i], w & 0xFFFFu);
            if (w >> 16) atomicAdd(&gj[2 * i + 1], w >> 16);
        }
        if (t < 256) {
            if (sm.exs[t]) atomicAdd(&ex[j * 512 + t], sm.exs[t]);
            if (sm.exf[t]) atomicAdd(&ex[j * 512 + 256 + t], sm.exf[t]);
        }
        __threadfence();
        __syncthreads();
        if (t == 0) sm.flag = (atomicAdd(&ex[1024 + j], 1u) == (unsigned)(S - 1));
        __syncthreads();
        if (!sm.flag) return;
        __threadfence();
        if (t < 256) {
            sm.exs[t] = __ldcg(&ex[j * 512 + t]); sm.exf[t] = __ldcg(&ex[j * 512 + 256 + t]);
            ex[j * 512 + t] = 0u; ex[j * 512 + 256 + t] = 0u;          // leave the workspace zeroed
        }
        if (t == 0) ex[1024 + j] = 0u;
    }
    // ---- totals per bin (shared + the 32768-count blocks already moved to global), marginals, entropy ----
    double sumT = 0.0;                                 // sum of c*log2(c) over this thread's bins
    uint32_t colacc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) colacc[k] = 0u;
#pragma unroll 1
    for (int rr = 0; rr < 8; ++rr) {
        const int row = warp + 32 * rr;
        uint32_t rsum = 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int wd = row * 128 + lane + 32 * k;
            uint2 g = __ldcg(reinterpret_cast<const uint2*>(gj + 2 * wd));
            if (fused) {
                const uint32_t w = sm.jh[wd];
                g.x += w & 0xFFFFu; g.y += w >> 16;
                *reinterpret_cast<uint2*>(gj + 2 * wd) = g;
            }
            rsum += g.x + g.y;
            colacc[2 * k] += g.x; colacc[2 * k + 1] += g.y;
            sumT += (g.x < (uint32_t)kClogN) ? sm.clog[g.x] : (double)g.x * log2((double)g.x);
            sumT += (g.y < (uint32_t)kClogN) ? sm.clog[g.y] : (double)g.y * log2((double)g.y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) rsum += __shfl_xor_sync(0xffffffffu, rsum, o);
        if (lane == 0) sm.rows[row] = rsum;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (colacc[2 * k]) atomicAdd(&sm.cols[2 * (lane + 32 * k)], colacc[2 * k]);
        if (colacc[2 * k + 1]) atomicAdd(&sm.cols[2 * (lane + 32 * k) + 1], colacc[2 * k + 1]);
    }
    __syncthreads();
    double v[5] = {0.0, 0.0, 0.0, sumT, 0.0};
    if (t < 256) {
        const uint32_t hs = sm.rows[t] + sm.exs[t], hf = sm.cols[t] + sm.exf[t];
        cn[j * 256 + t] = hs;
        if (j == 0) cn[512 + t] = hf;
        const double invP = 1.0 / (double)P;
        const double ps = hs * invP, pf = hf * invP;
        v[0] = hs ? -ps * log2(ps) : 0.0;                       // metric.py:119-125
        v[1] = hf ? -pf * log2(pf) : 0.0;
        v[2] = (hs && hf) ? ps * log2(ps / pf) : 0.0;           // metric.py:158-165
        v[4] = (double)sm.rows[t];
    }
    if (!ent) return;
    block_sum<5, kHT>(v, sm.red);
    if (t == 0) {
        double* e = ent + (size_t)n * estride;
        // joint entropy -sum p log2 p with p = c / P (metric.py:148-154) from sum c and sum c log2 c
        const double je = (log2((double)P) * v[4] - v[3]) / (double)P;
        const double mi = v[0] + v[1] - je;                     // metric.py:179-188
        e[j == 0 ? MMIF_EN_A : MMIF_EN_B] = v[0];
        e[j == 0 ? MMIF_JE_AF : MMIF_JE_BF] = je;
        e[j == 0 ? MMIF_CE_AF : MMIF_CE_BF] = v[2];
        e[j == 0 ? MMIF_MI_AF : MMIF_MI_BF] = mi;
        e[j == 0 ? MMIF_NMI_AF : MMIF_NMI_BF] = 2.0 * mi / (v[0] + v[1]);
        if (j == 0) { e[MMIF_EN_F] = v[1]; e[11] = 0.0; }
    }
}

size_t hist_extra_words(int N) { return (size_t)N * kHistExtraWords; }

int launch_hist(const float* a, const float* b, const float* f, int N, int H, int W, uint32_t* counts, double* ent,
                long long estride, MetricWs& ws, cudaStream_t st) {
    const long long P = (long long)H * W;
    // Pixel splits per (pair, joint): one CTA per SM, so 2 N S CTAs run in ceil(2 N S / 148) waves of (P / S pixels + the
    // merge of a split CTA's 65536 counters into the global histogram, worth ~kMergePx pixels of counting).  Minimise
    // waves x (P / S + merge): 32 pairs of 1224x1024 take S = 2 (128 CTAs, one wave) instead of 64 CTAs on 148 SMs.
    constexpr long long kMergePx = 180000;
    int S = 1;
    if (P >= 65536) {
        double best = 1e300;
        for (int c = 1; c <= 16; ++c) {
            const long long ctas = 2ll * N * c;
            const double waves = (double)((ctas + 147) / 148);
            const double cost = waves * ((double)P / c + (c > 1 ? (double)kMergePx : 0.0));
            if (cost < best * 0.97) { best = cost; S = c; }      // a split must pay for itself by > 3 %
        }
    }
    static const char* force = getenv("MMIF_HIST_SPLIT");        // tuning aid (tools/hist_split_scan.py)
    if (force && atoi(force) >= 1 && atoi(force) <= 16) S = atoi(force);
    static unsigned long long attr_done = 0ull;
    if (first_use_on_device(&attr_done)) {
        MMIF_CUDA(cudaFuncSetAttribute(hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HistSmem)));
    }
    dim3 grid(2 * S, N);
    hist_kernel<<<grid, kHT, sizeof(HistSmem), st>>>(a, b, f, P, S, counts, ws.hist_extra, ent, estride);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// =============================================================================== TVLoss
__global__ void __launch_bounds__(256)
tv_kernel(const float* __restrict__ X, int H, int W, int rpb, int norm, float weight, long long NI, double* partial,
          unsigned* counters, double* out) {
    __shared__ double red[2 * 8];
    __shared__ int flag;
    const int n = blockIdx.y, blk = blockIdx.y * gridDim.x + blockIdx.x, nblk = gridDim.x * gridDim.y;
    const float* x = X + (size_t)n * H * W;
    const int r0 = blockIdx.x * rpb, r1 = min(r0 + rpb, H);
    double acc[2] = {0.0, 0.0};
    for (int c = threadIdx.x; c < W; c += 256) {
        float sv = 0.f, sh = 0.f;
        for (int r = r0; r < r1; ++r) {
            const size_t p = (size_t)r * W + c;
            const float v = __ldg(x + p);
            if (r + 1 < H) sv += norm_val(__ldg(x + p + W) - v, norm);
            if (c + 1 < W) sh += norm_val(__ldg(x + p + 1) - v, norm);
        }
        acc[0] += sv; acc[1] += sh;
    }
    double t[2];
    // all images reduce into one scalar: use sample slot 0 with nblk = whole grid
    if (!block_finish<2, 256>(acc, red, &flag, partial, counters, 0, blk, nblk, t)) return;
    out[0] = (double)weight * (t[0] / ((double)NI * (H - 1) * W) + t[1] / ((double)NI * H * (W - 1)));   // loss.py:354-358
}

int launch_tv(const float* x, int N, int H, int W, int norm, float weight, double* out, MetricWs& ws, cudaStream_t st) {
    if (H < 2 || W < 2) { set_error("tv: H and W must be >= 2"); return MMIF_E_SHAPE; }
    const int rpb = stats_rows_per_block(N, H);
    dim3 grid(ceil_div(H, rpb), N);
    tv_kernel<<<grid, 256, 0, st>>>(x, H, W, rpb, norm, weight, (long long)N, ws.partial, ws.counters, out);
    mmif::count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

}  // namespace mmif
