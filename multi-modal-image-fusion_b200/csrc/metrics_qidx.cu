// Window-based fusion quality indices: Piella & Heijmans' Q / Q_W / Q_E (ICIP 2003) and Yang et al.'s Q_Y (Information
// Fusion 2008).  Definitions: oracle/quality_index.py.
//
// One launch covers N pairs and reads a, b and f once.  CTA (strip, segment, pair) owns kQT = 128 window columns and
// kQRows window rows (a window is named by its top-left pixel; the 8x8 box windows and the 11x11 Gaussian windows share
// that grid):
//   * the input tile, rows r0-1 .. r0+kQRows+9 and columns c0-1 .. c0+138 of a, b, f, lands in shared memory with the
//     reflect border of metric.py:192-206 (pixel -1 is pixel 1, pixel H is pixel H-2);
//   * the Sobel magnitudes of the three images (Q_E) are formed from that tile into shared memory; they never reach HBM;
//   * per window row: a V-pass (thread = column) forms the 8-row box sums of the 8 moment products of (a,f), (b,f) on the
//     images and on the edge images, and the 11-tap Gaussian sums of the 9 products of (a,f), (b,f), (a,b); an H-pass
//     (thread = window column) sums 8 box / 11 Gaussian columns and hands the moments to the window's index terms.
// Moments are taken of shifted data x - c (c = the tile's minimum, per image) so E[x^2] - mu^2 does not cancel in fp32;
// the box sums of integer images are exact.  Each window's terms are formed and accumulated in double; per-CTA partials
// are re-reduced in a fixed order by the last CTA of the pair (block_finish): deterministic, no float atomics.
#include "metrics.cuh"

namespace mmif {
namespace {

constexpr int kQT = 128;                    // threads per CTA = window columns per strip
constexpr int kQRows = 16;                  // window rows per CTA
constexpr int kBox = 8;                     // Piella box window
constexpr int kQyWin = 11;                  // Yang: the metric SSIM window
constexpr int kTileR = kQRows + kQyWin;     // input rows r0-1 .. r0+kQRows+9
constexpr int kTileC = kQT + kQyWin + 1;    // input columns c0-1 .. c0+kQT+9 (+1 pad)
constexpr int kEdgeR = kQRows + kBox - 1;   // Sobel rows r0 .. r0+kQRows+6
constexpr int kEdgeC = kQT + kBox;          // Sobel columns c0 .. c0+kQT+6 (+1 pad)
constexpr int kVCol = kQT + kQyWin - 1;     // V-pass columns (the Gaussian H-pass reads kQT + 10)
constexpr int kBoxMaps = 8;                 // Sa Sb Sf Saa Sbb Sff Saf Sbf
constexpr int kGMaps = 9;                   // the same + Sab
constexpr int kQK = 7;                      // per-pair sums, see below

struct QSmem {
    float img[3][kTileR][kTileC];
    float edge[3][kEdgeR][kEdgeC];
    float vbox[2][kBoxMaps][kVCol];         // [images, edge images]
    float vg[kGMaps][kVCol];
    double red[kQK * (kQT / 32)];
    float shift[6 * (kQT / 32)];
    int flag;
};

__device__ __forceinline__ int reflect_clamp(int x, int n) {
    x = (x < 0) ? -x : x;
    x = (x >= n) ? 2 * n - 2 - x : x;
    return min(max(x, 0), n - 1);
}

// Wang-Bovik universal index with img_qi.m's degenerate branches.
__device__ __forceinline__ double q0(double mx, double my, double vx, double vy, double cxy) {
    const double vs = vx + vy, ms = mx * mx + my * my;
    if (vs == 0.0) return ms == 0.0 ? 1.0 : 2.0 * mx * my / ms;
    if (ms == 0.0) return 2.0 * cxy / vs;
    return 4.0 * cxy * mx * my / (vs * ms);
}
__device__ __forceinline__ double lambda_of(double sa, double sb) { return (sa + sb == 0.0) ? 0.5 : sa / (sa + sb); }

// Piella terms of one box window from its shifted sums s[8] (see kBoxMaps) and the shifts c[3]:
// acc[0] += term, acc[1] += C * term, acc[2] += C.
__device__ __forceinline__ void piella_window(const float (&s)[kBoxMaps], const float (&c)[3], double* acc) {
    constexpr double k = 1.0 / (kBox * kBox);
    const double ma = s[0] * k, mb = s[1] * k, mf = s[2] * k;
    const double va = fmax(s[3] * k - ma * ma, 0.0), vb = fmax(s[4] * k - mb * mb, 0.0), vf = fmax(s[5] * k - mf * mf, 0.0);
    const double caf = s[6] * k - ma * mf, cbf = s[7] * k - mb * mf;
    const double Ma = ma + c[0], Mb = mb + c[1], Mf = mf + c[2];
    const double lam = lambda_of(va, vb);
    const double term = lam * q0(Ma, Mf, va, vf, caf) + (1.0 - lam) * q0(Mb, Mf, vb, vf, cbf);
    const double C = fmax(va, vb);
    acc[0] += term;
    acc[1] += C * term;
    acc[2] += C;
}

__global__ void __launch_bounds__(kQT, 2)
quality_index_kernel(const float* __restrict__ A, const float* __restrict__ Bm, const float* __restrict__ F, int H, int W,
                     Taps tp, double C1, double C2, double* partial, unsigned* counters, double* out) {
    extern __shared__ __align__(16) unsigned char qidx_smem_raw[];
    QSmem& sm = *reinterpret_cast<QSmem*>(qidx_smem_raw);
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int n = blockIdx.z, blk = blockIdx.y * gridDim.x + blockIdx.x, nblk = gridDim.x * gridDim.y;
    const int c0 = blockIdx.x * kQT, r0 = blockIdx.y * kQRows;
    const size_t off = (size_t)n * H * W;
    const float* src[3] = {A + off, Bm + off, F + off};

    // ---- input tile with the reflect border; running minimum of the finite values per image ----
    float mn[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) mn[k] = 3.0e38f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        for (int i = t; i < kTileR * kTileC; i += kQT) {
            const int tr = i / kTileC, tc = i - tr * kTileC;
            const int r = reflect_clamp(r0 - 1 + tr, H), c = reflect_clamp(c0 - 1 + tc, W);
            const float v = __ldg(src[k] + (size_t)r * W + c);
            sm.img[k][tr][tc] = v;
            if (fabsf(v) <= 3.0e38f) mn[k] = fminf(mn[k], v);
        }
    }
    __syncthreads();
    // ---- Sobel magnitudes (metric.py:192-206), IEEE fp32 like the reference's conv2d + pow(0.5) ----
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        for (int i = t; i < kEdgeR * kEdgeC; i += kQT) {
            const int er = i / kEdgeC, ec = i - er * kEdgeC;
            const float(*x)[kTileC] = sm.img[k];
            const int tr = er + 1, tc = ec + 1;
            const float dU = x[tr - 1][tc + 1] - x[tr - 1][tc - 1], dM = x[tr][tc + 1] - x[tr][tc - 1],
                        dD = x[tr + 1][tc + 1] - x[tr + 1][tc - 1];
            const float sU = x[tr - 1][tc - 1] + 2.f * x[tr - 1][tc] + x[tr - 1][tc + 1];
            const float sD = x[tr + 1][tc - 1] + 2.f * x[tr + 1][tc] + x[tr + 1][tc + 1];
            const float gx = dU + 2.f * dM + dD, gy = sD - sU;
            const float g = __fsqrt_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)));
            sm.edge[k][er][ec] = g;
            if (fabsf(g) <= 3.0e38f) mn[3 + k] = fminf(mn[3 + k], g);
        }
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
        if (lane == 0) sm.shift[warp * 6 + k] = mn[k];
    }
    __syncthreads();
    float cs[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        float m = sm.shift[k];
#pragma unroll
        for (int w = 1; w < kQT / 32; ++w) m = fminf(m, sm.shift[w * 6 + k]);
        cs[k] = (m < 3.0e38f) ? m : 0.f;
    }
    const float ci[3] = {cs[0], cs[1], cs[2]}, ce[3] = {cs[3], cs[4], cs[5]};
    const double s = tp.wsum, eps = tp.weps;

    // acc: 0 sum term, 1 sum C term, 2 sum C (images); 3 sum term', 4 sum C' term', 5 sum C' (edge images); 6 sum Q_Y term
    double acc[kQK];
#pragma unroll
    for (int k = 0; k < kQK; ++k) acc[k] = 0.0;
    const int j = c0 + t;
    const bool col_box = j <= W - kBox, col_g = j <= W - kQyWin;
    for (int ii = 0; ii < kQRows && r0 + ii <= H - kBox; ++ii) {
        // ---- V-pass: thread = column (two passes cover the kVCol columns) ----
        for (int col = t; col < kVCol; col += kQT) {
            if (col < kEdgeC - 1) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    float v[kBoxMaps];
#pragma unroll
                    for (int m = 0; m < kBoxMaps; ++m) v[m] = 0.f;
#pragma unroll
                    for (int k = 0; k < kBox; ++k) {
                        const float* cc = g ? ce : ci;
                        const float xa = (g ? sm.edge[0][ii + k][col] : sm.img[0][ii + k + 1][col + 1]) - cc[0];
                        const float xb = (g ? sm.edge[1][ii + k][col] : sm.img[1][ii + k + 1][col + 1]) - cc[1];
                        const float xf = (g ? sm.edge[2][ii + k][col] : sm.img[2][ii + k + 1][col + 1]) - cc[2];
                        v[0] += xa; v[1] += xb; v[2] += xf;
                        v[3] = fmaf(xa, xa, v[3]); v[4] = fmaf(xb, xb, v[4]); v[5] = fmaf(xf, xf, v[5]);
                        v[6] = fmaf(xa, xf, v[6]); v[7] = fmaf(xb, xf, v[7]);
                    }
#pragma unroll
                    for (int m = 0; m < kBoxMaps; ++m) sm.vbox[g][m][col] = v[m];
                }
            }
            float v[kGMaps];
#pragma unroll
            for (int m = 0; m < kGMaps; ++m) v[m] = 0.f;
#pragma unroll
            for (int k = 0; k < kQyWin; ++k) {
                const float w = tp.w[k];
                const float xa = sm.img[0][ii + k + 1][col + 1] - ci[0];
                const float xb = sm.img[1][ii + k + 1][col + 1] - ci[1];
                const float xf = sm.img[2][ii + k + 1][col + 1] - ci[2];
                const float wa = w * xa, wb = w * xb, wf = w * xf;
                v[0] += wa; v[1] += wb; v[2] += wf;
                v[3] = fmaf(wa, xa, v[3]); v[4] = fmaf(wb, xb, v[4]); v[5] = fmaf(wf, xf, v[5]);
                v[6] = fmaf(wa, xf, v[6]); v[7] = fmaf(wb, xf, v[7]); v[8] = fmaf(wa, xb, v[8]);
            }
#pragma unroll
            for (int m = 0; m < kGMaps; ++m) sm.vg[m][col] = v[m];
        }
        __syncthreads();
        // ---- H-pass: thread = window column ----
        const int i = r0 + ii;
        if (col_box) {
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                float sb[kBoxMaps];
#pragma unroll
                for (int m = 0; m < kBoxMaps; ++m) {
                    float a = 0.f;
#pragma unroll
                    for (int k = 0; k < kBox; ++k) a += sm.vbox[g][m][t + k];
                    sb[m] = a;
                }
                piella_window(sb, g ? ce : ci, acc + 3 * g);
            }
        }
        if (col_g && i <= H - kQyWin) {
            float mg[kGMaps];
#pragma unroll
            for (int m = 0; m < kGMaps; ++m) {
                float a = 0.f;
#pragma unroll
                for (int k = 0; k < kQyWin; ++k) a = fmaf(tp.w[k], sm.vg[m][t + k], a);
                mg[m] = a;
            }
            // reference statistics of the 2-D window that sums to s = 1 + eps (stencil.cuh, Shift):
            // mu = mu' + s c, var = E'[x'^2] - mu'^2 - eps c (2 mu' + s c), cov = E'[x'y'] - mu_x' mu_y' - eps (c_x mu_y' + c_y mu_x' + s c_x c_y)
            double mu[3], var[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double m = mg[k], c = ci[k];
                mu[k] = m + s * c;
                var[k] = fmax((double)mg[3 + k] - m * m - eps * c * (2.0 * m + s * c), 0.0);
            }
            auto cov = [&](int x, int y, float e) {
                const double mx = mg[x], my = mg[y], cx = ci[x], cy = ci[y];
                return (double)e - mx * my - eps * (cx * my + cy * mx + s * cx * cy);
            };
            auto ssim = [&](int x, int y, double cxy) {
                return ((2.0 * mu[x] * mu[y] + C1) * (2.0 * cxy + C2)) /
                       ((mu[x] * mu[x] + mu[y] * mu[y] + C1) * (var[x] + var[y] + C2));
            };
            const double saf = ssim(0, 2, cov(0, 2, mg[6])), sbf = ssim(1, 2, cov(1, 2, mg[7]));
            const double sab = ssim(0, 1, cov(0, 1, mg[8]));
            const double lam = lambda_of(var[0], var[1]);
            acc[6] += (sab >= 0.75) ? lam * saf + (1.0 - lam) * sbf : fmax(saf, sbf);
        }
        __syncthreads();
    }

    double tot[kQK];
    if (!block_finish<kQK, kQT>(acc, sm.red, &sm.flag, partial, counters, n, blk, nblk, tot)) return;
    const double nbox = (double)(H - kBox + 1) * (double)(W - kBox + 1);
    const double ng = (double)(H - kQyWin + 1) * (double)(W - kQyWin + 1);
    double* o = out + (size_t)n * MMIF_QIDX_DOUBLES;
    const double q = tot[0] / nbox;
    const double qw = (tot[2] == 0.0) ? q : tot[1] / tot[2];
    const double qw_e = (tot[5] == 0.0) ? tot[3] / nbox : tot[4] / tot[5];
    o[MMIF_QIDX_Q] = q;
    o[MMIF_QIDX_QW] = qw;
    o[MMIF_QIDX_QE] = qw * qw_e;
    o[MMIF_QIDX_QY] = tot[6] / ng;
    o[MMIF_QIDX_SUM_TERM] = tot[0];
    o[MMIF_QIDX_BOX_WINDOWS] = nbox;
    o[MMIF_QIDX_SUM_CTERM] = tot[1];
    o[MMIF_QIDX_SUM_C] = tot[2];
    o[MMIF_QIDX_SUM_TERM_E] = tot[3];
    o[MMIF_QIDX_SUM_CTERM_E] = tot[4];
    o[MMIF_QIDX_SUM_C_E] = tot[5];
    o[MMIF_QIDX_SUM_TERM_Y] = tot[6];
    o[MMIF_QIDX_QY_WINDOWS] = ng;
}

struct QGeom {
    dim3 grid;
    size_t counter_bytes, partial_bytes;
};
QGeom qidx_geom(int N, int H, int W) {
    QGeom g;
    g.grid = dim3(ceil_div(W - kBox + 1, kQT), ceil_div(H - kBox + 1, kQRows), N);
    g.counter_bytes = ((size_t)N * sizeof(unsigned) + 255) & ~(size_t)255;
    g.partial_bytes = (size_t)N * g.grid.x * g.grid.y * kQK * sizeof(double);
    return g;
}
bool qidx_shape_ok(int N, int H, int W) { return N >= 1 && H >= kQyWin && W >= kQyWin && (long long)N * H * W < (1ll << 40); }

}  // namespace
}  // namespace mmif

using namespace mmif;

extern "C" size_t mmif_quality_index_workspace_bytes(int N, int H, int W) {
    if (!qidx_shape_ok(N, H, W)) return 0;
    const QGeom g = qidx_geom(N, H, W);
    return g.counter_bytes + g.partial_bytes;
}

extern "C" int mmif_quality_index(const float* a, const float* b, const float* f, int N, int H, int W, double* out, void* ws,
                                  size_t ws_bytes, void* stream) {
    if (!a || !b || !f || !out) { set_error("quality_index: null image or out pointer"); return MMIF_E_NULL; }
    if (!qidx_shape_ok(N, H, W)) { set_error("quality_index: bad shape (%d,%d,%d): N >= 1, H and W >= 11", N, H, W); return MMIF_E_SHAPE; }
    if ((((uintptr_t)a | (uintptr_t)b | (uintptr_t)f) & 3) || (((uintptr_t)out | (uintptr_t)ws) & 7)) {
        set_error("quality_index: image pointers must be 4-byte, out and ws 8-byte aligned");
        return MMIF_E_ALIGN;
    }
    const QGeom g = qidx_geom(N, H, W);
    if (!ws || ws_bytes < g.counter_bytes + g.partial_bytes) {
        set_error("quality_index: workspace of %zu bytes, %zu needed", ws_bytes, g.counter_bytes + g.partial_bytes);
        return MMIF_E_WORKSPACE;
    }
    static unsigned long long attr_done = 0ull;
    if (first_use_on_device(&attr_done)) {
        MMIF_CUDA(cudaFuncSetAttribute(quality_index_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(QSmem)));
    }
    Taps tp;
    make_taps(&tp, kQyWin, 1.5);
    const double C1 = (0.01 * 255.0) * (0.01 * 255.0), C2 = (0.03 * 255.0) * (0.03 * 255.0);
    unsigned char* w = static_cast<unsigned char*>(ws);
    quality_index_kernel<<<g.grid, kQT, sizeof(QSmem), (cudaStream_t)stream>>>(
        a, b, f, H, W, tp, C1, C2, reinterpret_cast<double*>(w + g.counter_bytes), reinterpret_cast<unsigned*>(w), out);
    count_launch(MMIF_CNT_METRIC);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
