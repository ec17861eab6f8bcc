/*
 * mmif_b200.h — C ABI of libmmif_b200.so: the fusion objective (reference core/loss.py)
 * and the objective metric suite (reference core/metric.py) as sm_100a CUDA kernels.
 *
 * The reference repository is pure Python and has no FFI; the boundary it defines is the
 * Python call surface (core/loss.py:16-19, core/metric.py:16-21).  Every entry point below
 * names the reference function(s) it replaces.  The Python mirror of that surface
 * (multi-modal-image-fusion_b200/core/{loss,metric}.py) binds these symbols with ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every image pointer is DEVICE memory, dense row-major
 *     float32 [N][H][W] (the reference's (N,1,H,W) tensors, C == 1);
 *   - return 0 on success, negative MMIF_E_* on error; mmif_last_error() gives the text for the
 *     calling thread; no exception, abort or device synchronisation crosses the ABI;
 *   - the caller owns every buffer, including the workspace `ws` (size from the matching
 *     *_workspace_bytes call; 256-byte aligned; must be zero-filled once before its first use
 *     WITH A GIVEN SHAPE — the kernels leave their counters zeroed again, but the carve-up
 *     depends on the shape, so re-zero it (or use another buffer) when the shape changes; one
 *     workspace serves one stream at a time); the library never allocates or frees device memory;
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it and results stay on the
 *     device; re-entrant (no mutable globals besides __constant__ tap tables written per launch
 *     configuration under a mutex).
 */
#ifndef MMIF_B200_H_
#define MMIF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMIF_VERSION 100 /* 0.1.0 */

enum {
    MMIF_OK = 0,
    MMIF_E_NULL = -1,        /* null pointer argument */
    MMIF_E_SHAPE = -2,       /* unsupported shape (e.g. H or W smaller than the window) */
    MMIF_E_MODE = -3,        /* unsupported mode / configuration value */
    MMIF_E_WORKSPACE = -4,   /* workspace too small */
    MMIF_E_ALIGN = -5,       /* pointer not 4-byte aligned */
    MMIF_E_CUDA = -6,        /* a CUDA runtime call failed (text in mmif_last_error) */
    MMIF_E_DEVICE = -7       /* not an sm_100 device / no device */
};

enum { MMIF_COMBINE_MAX = 0, MMIF_COMBINE_AVG = 1 };   /* PixelLoss/GradLoss forward(mode=) loss.py:294-304,330-344 */
enum { MMIF_NORM_L1 = 1, MMIF_NORM_L2 = 2 };           /* NormLoss mode, loss.py:375-385 */

/* Configuration of the three-term objective as train.py:302-317 wires it. */
typedef struct MmifLossCfg {
    float w_ssim;       /* SSIMLoss weight   (train.py:306, 1.0)  */
    float w_pixel;      /* PixelLoss weight  (train.py:307, 0.01) */
    float w_grad;       /* GradLoss weight   (train.py:308, 0.1)  */
    float data_range;   /* L of C1=(0.01L)^2, C2=(0.03L)^2 (loss.py:91-93); SSIMLoss default 1.0 */
    int32_t pixel_combine; /* MMIF_COMBINE_*  */
    int32_t grad_combine;  /* MMIF_COMBINE_*  */
    int32_t pixel_norm;    /* MMIF_NORM_*     */
    int32_t grad_norm;     /* MMIF_NORM_*     */
    int32_t want_grad;     /* fwd only: !=0 -> single-pass variant: the same launch also writes
                              d(l_ssim + l_pixel + l_grad)/d(imgf) (unit upstream gradients, the
                              weights above applied) into `dF_unit`; else ignored.  2 = the same for a
                              caller that reads the three loss values only (the training step,
                              train.py:64-71): of the per-sample block the SSIM means are written, the
                              cs / sigma entries are 0 (their sums cost 1.2 % of the kernel) */
    int32_t reserved;
} MmifLossCfg;

/* Layout of the double[] written by mmif_fusion_loss_fwd (device memory). */
enum {
    MMIF_LOSS_SSIM = 0,   /* w_ssim * (1 - (mean_b ssim(I1,If) + mean_b ssim(I2,If))/2)   SSIMLoss('ssim') loss.py:253-257,284 */
    MMIF_LOSS_PIXEL = 1,  /* PixelLoss value                                               loss.py:294-304 */
    MMIF_LOSS_GRAD = 2,   /* GradLoss value                                                loss.py:330-344 */
    MMIF_LOSS_TOTAL = 3,  /* sum of the three (train.py:69) */
    MMIF_LOSS_HEAD = 4,   /* per-sample block starts here: B x MMIF_LOSS_PER_SAMPLE */
    MMIF_LOSS_PER_SAMPLE = 6 /* ssim1, cs1, sigma1, ssim2, cs2, sigma2 — the dict of SSIM.forward (loss.py:105-110) */
};

/* Launch bookkeeping (host side, process-wide, monotonically increasing): which kernels the library has enqueued.
 * Lets a caller (and the parity tests) verify WHICH path served a call — e.g. that SSIMLoss + PixelLoss + GradLoss
 * with a gradient wanted ran the single-pass loss+gradient kernel — and is what bench.py's `gpu_launches` counts. */
enum {
    MMIF_CNT_LOSS_FWD = 0,         /* moment_fwd_kernel<11, SSIM> with the pixel / Sobel terms: forward of the two-kernel path */
    MMIF_CNT_LOSS_SINGLE_PASS = 1, /* fusion_loss_bwd_kernel<11, *, ZMODE=1, 0>: loss values AND dL/dIf in one launch */
    MMIF_CNT_LOSS_BWD = 2,         /* fusion_loss_bwd_kernel<11, *, 0, 0>: recomputing backward */
    MMIF_CNT_RESCALE = 3,          /* rescale_unit_kernel (backward of the single-pass path) */
    MMIF_CNT_SSIM_BWD_EXT = 4,     /* SSIM-only backward launches (w-ssim, MS-SSIM levels, MSW-SSIM windows, SSIM dict) */
    MMIF_CNT_MOMENT_FWD = 5,       /* every other moment_fwd_kernel launch (SSIM windows, maps, VIF scales, MSW) */
    MMIF_CNT_METRIC = 6,           /* metric-suite kernels other than moment_fwd (pixel metrics, histograms, pyramids) */
    MMIF_CNT_AUX = 7,              /* small operators: pad / halve / widen / norm / tv and their adjoints */
    MMIF_CNT_TMAP_ENCODE = 8,      /* cuTensorMapEncodeTiled calls (not a launch) */
    MMIF_CNT_TMAP_HIT = 9,         /* tensor maps served from the per-thread memo (not a launch) */
    MMIF_CNT_TMAP_FAIL = 10,       /* encodings the driver refused although shape and alignment qualify (should stay 0) */
    MMIF_CNT_N = 16
};
/* out[i] = counter i for i < n (HOST memory). */
int mmif_launch_counts(unsigned long long* out, int n);

/* Diagnostic (host only, no launch): how the loss + gradient kernels cut a (B, H, W) problem into CTAs.  kernel = 0: the
 * 2-CTA kernel, 1: the warp-specialised kernel.  out[10] = {nstrip, nseg, n_tall, seg_rows, seg_short, fine_strips, fine_rows,
 * nseg_fine, CTAs per sample, gradient columns per strip}; the tests check that every (row, column) is owned exactly once. */
int mmif_loss_geometry(int B, int H, int W, int kernel, int* out10);

int mmif_version(void);
const char* mmif_last_error(void);
/* 0 if device `dev` is usable by this library (compute capability 10.x). */
int mmif_check_device(int dev);
/* Register the reference's own 1-D Gaussian taps for (win, sigma): `taps` = win HOST floats, i.e.
 * _gaussian_kernel(win, sigma) of loss.py:24-30 / metric.py:290-296 evaluated by the caller with
 * the reference's torch ops.  Optional: without it the library builds the table itself (float32
 * taps normalised by a sequentially accumulated float32 sum), which can differ from torch's table
 * in the last bit of the normalisation.  win <= 17.  Thread-safe; affects later launches. */
int mmif_set_gaussian_taps(int win, double sigma, const float* taps);

/* ---------------------------------------------------------------- fusion objective ------- */
size_t mmif_loss_workspace_bytes(int B, int H, int W);
size_t mmif_loss_out_doubles(int B);

/* Replaces SSIMLoss('ssim').forward + PixelLoss.forward + GradLoss.forward (loss.py:252-257,
 * 294-304, 330-344) and the SSIM.forward dict (loss.py:179-185) in one launch.
 * i1,i2,f: [B][H][W]; out: mmif_loss_out_doubles(B) doubles = the MMIF_LOSS_* block of 4 + 6 B doubles followed by
 * its float32 mirror (same indices, at (float*)(out + 4 + 6 B)); dF_unit: [B][H][W] or NULL. */
int mmif_fusion_loss_fwd(const float* i1, const float* i2, const float* f, int B, int H, int W,
                         const MmifLossCfg* cfg, double* out, float* dF_unit,
                         void* ws, size_t ws_bytes, void* stream);

/* Replaces autograd's backward of the three modules w.r.t. imgf (train.py:71): recomputes the
 * stencil and writes dF = g[0]*w_ssim*dLssim/dIf + g[1]*w_pixel*dLpixel/dIf + g[2]*w_grad*dLgrad/dIf.
 * gout3: 3 floats in DEVICE memory (upstream gradients of the three loss values).
 * dF_unit: NULL, or the buffer a want_grad forward (same inputs, same cfg) filled.  When it is given
 * and the three upstream gradients are equal (total = l1 + l2 + l3, train.py:69) the kernel only
 * rescales it (8 B/pixel); otherwise it recomputes.  The decision is taken on the device.
 * dF may alias dF_unit: the rescale then happens in place and costs nothing when the common upstream
 * gradient is exactly 1 (total.backward()); the buffer no longer holds the unit gradient afterwards. */
int mmif_fusion_loss_bwd(const float* i1, const float* i2, const float* f, int B, int H, int W,
                         const MmifLossCfg* cfg, const float* gout3, const float* dF_unit, float* dF,
                         void* ws, size_t ws_bytes, void* stream);

/* The same, with the three upstream gradients as separate DEVICE scalars exactly as autograd hands them to the node
 * (train.py:69-71: total = l1 + l2 + l3; total.backward()).  A NULL pointer means that loss value received no
 * gradient (0); at least one must be non-NULL. */
int mmif_fusion_loss_bwd3(const float* i1, const float* i2, const float* f, int B, int H, int W,
                          const MmifLossCfg* cfg, const float* g_ssim, const float* g_pixel, const float* g_grad,
                          const float* dF_unit, float* dF, void* ws, size_t ws_bytes, void* stream);

/* d/dIf of  scale * sum_n sum_k pair_w[n][k] * mean_windows(S_k)(I_k[n], If[n]),  S = ssim or (cs_only) the
 * contrast-structure term, times the device scalar gout1[0].  pair_w: [B][2] device floats or NULL (= 1).
 * Building block of SSIMLoss('w-ssim') (loss.py:259-266: per-sample gamma from the sources) and of the
 * MS-SSIM levels (loss.py:140-158: cs on levels 0..3, ssim on level 4, per-sample chain-rule factors). */
int mmif_ssim_bwd_ex(const float* i1, const float* i2, const float* f, int B, int H, int W, float data_range,
                     const float* gout1, const float* pair_w, int cs_only, float scale, float* dF,
                     void* ws, size_t ws_bytes, void* stream);

/* SSIM(win_size) of the loss module (loss.py:163-185 -> calc_ssim, loss.py:52-110, size_average=True) for a window of
 * 11, 9, 7, 5 or 3 taps (sigma by the loss rule, loss.py:34): mmif_ssim_fwd_win writes the per-sample means
 * ssim, cs, sigma of the pairs (i1, f), (i2, f) in the loss block layout (out: mmif_loss_out_doubles(B) doubles);
 * mmif_ssim_bwd_ex_win is mmif_ssim_bwd_ex with that window.  ws from mmif_loss_workspace_bytes. */
int mmif_ssim_fwd_win(const float* i1, const float* i2, const float* f, int B, int H, int W, int win, float data_range,
                      double* out, void* ws, size_t ws_bytes, void* stream);
int mmif_ssim_bwd_ex_win(const float* i1, const float* i2, const float* f, int B, int H, int W, int win, float data_range,
                         const float* gout1, const float* pair_w, int cs_only, float scale, float* dF,
                         void* ws, size_t ws_bytes, void* stream);

/* Generic calc_ssim of the loss module (loss.py:52-110) for ONE pair (x, y) and ANY window of 1..17 taps (odd or even; the
 * taps of (win, sigma) as registered with mmif_set_gaussian_taps, else built by the library), with everything the
 * reference's autograd provides.  Direct k x k evaluation in double: the slow, complete companion of the strip kernels.
 *   fwd: per_sample3 = [B][3] doubles (mean ssim, cs, sigma) or NULL; map_* = [B][H-win+1][W-win+1] floats or NULL
 *        (size_average=False).  ws: mmif_ssim_generic_workspace_bytes, zero-filled once (only needed with per_sample3).
 *   bwd: upstream gradients of ssim / cs / sigma as [B] floats (maps == 0, the per-sample means) or as per-position maps
 *        (maps != 0); any of the three may be NULL (= 0).  Writes d/dx and / or d/dy ([B][H][W] floats, either may be
 *        NULL).  coef: mmif_ssim_generic_coef_doubles doubles of device scratch. */
size_t mmif_ssim_generic_workspace_bytes(int B, int H, int W, int win);
size_t mmif_ssim_generic_coef_doubles(int B, int H, int W, int win);
int mmif_ssim_generic_fwd(const float* x, const float* y, int B, int H, int W, int win, double sigma, float data_range,
                          double* per_sample3, float* map_ssim, float* map_cs, float* map_sigma,
                          void* ws, size_t ws_bytes, void* stream);
int mmif_ssim_generic_bwd(const float* x, const float* y, int B, int H, int W, int win, double sigma, float data_range,
                          const float* g_ssim, const float* g_cs, const float* g_sigma, int maps, float* dx, float* dy,
                          double* coef, void* stream);

/* One window size (11, 9, 7, 5 or 3; sigma by the loss rule, loss.py:34) of MSW_SSIM.forward
 * (loss.py:226-237): out_sums8[8*n] = sum over window positions of gamma*ssim(I1,If) + (1-gamma)*ssim(I2,If),
 * gamma = sigma1/(sigma1+sigma2) per position.  mmif_mswssim_bwd: dF (+)= gout1[0] * scale *
 * d( sum_n out_sums8[8n] / (Hout*Wout) )/dIf;  ws from mmif_loss_workspace_bytes. */
int mmif_mswssim_fwd(const float* i1, const float* i2, const float* f, int B, int H, int W, int win, float data_range,
                     double* out_sums8, void* ws, size_t ws_bytes, void* stream);
int mmif_mswssim_bwd(const float* i1, const float* i2, const float* f, int B, int H, int W, int win, float data_range,
                     const float* gout1, float scale, int accumulate, float* dF, void* ws, size_t ws_bytes, void* stream);

/* MS-SSIM level step of the loss (loss.py:147-153): reflect-pad the odd edge, 2x2 mean; dst is
 * [N][(H+1)/2][(W+1)/2].  mmif_halve_bwd ACCUMULATES the adjoint into g_src. */
int mmif_halve(const float* src, int N, int H, int W, float* dst, void* stream);
int mmif_halve_bwd(const float* g_dst, int N, int H, int W, float* g_src_accum, void* stream);

/* F.pad(img, (p,p,p,p), 'reflect') of use_padding=True (loss.py:45-47) and its adjoint (writes g_src). */
int mmif_reflect_pad(const float* src, int N, int H, int W, int pad, float* dst, void* stream);
int mmif_reflect_pad_bwd(const float* g_dst, int N, int H, int W, int pad, float* g_src, void* stream);

/* TVLoss.forward (loss.py:347-358) on x [N][H][W]: out[0] = w*(norm(dv) + norm(dh)). */
int mmif_tv_loss(const float* x, int N, int H, int W, int norm, float weight, double* out,
                 void* ws, size_t ws_bytes, void* stream);

/* Backward of TVLoss (loss.py:347-358): gx = gout1[0] * d(tv)/dx, x and gx [N][H][W]. */
int mmif_tv_loss_bwd(const float* x, int N, int H, int W, int norm, float weight, const float* gout1, float* gx,
                     void* stream);

/* size_average=False of calc_ssim (reference loss.py:52-110 / metric.py:316-364): SSIM, CS and clamp(sigma1^2, 1e-4)
 * MAPS of the pairs (i1, f), (i2, f), each [B][H-10][W-10]; any of the six outputs may be NULL.  11-tap window.
 * ws from mmif_loss_workspace_bytes. */
int mmif_ssim_maps(const float* i1, const float* i2, const float* f, int B, int H, int W, float data_range,
                   float* ssim1, float* cs1, float* sigma1, float* ssim2, float* cs2, float* sigma2,
                   void* ws, size_t ws_bytes, void* stream);

/* test.py:49-73 post-step (SURVEY 8(f).4) in one pass over imgf: out = the loss block of mmif_fusion_loss_fwd
 * (mmif_loss_out_doubles(B) doubles; per sample ssim1, cs1, sigma1, ssim2, cs2, sigma2 = calc_ssim(i1, f) and
 * calc_ssim(i2, f) with `data_range`, test.py:51-52) and, if denorm_u8 != NULL, the image save_result / denorm write
 * (common.py:74-81, data/transform.py:32-35): uint8(clip(f, 0, 1) * 255) as [B][H][W] bytes. */
int mmif_test_post(const float* i1, const float* i2, const float* f, int B, int H, int W, float data_range,
                   double* out, unsigned char* denorm_u8, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- metric suite ----------- */
/* All metric entries are batched over N independent pairs (a[n], b[n], f[n]) of one shape and
 * write doubles per pair.  ws from mmif_metric_workspace_bytes. */
size_t mmif_metric_workspace_bytes(int N, int H, int W);

enum { /* mmif_stats output, per pair */
    MMIF_ST_MEAN_F = 0, /* calc_mean(f)   metric.py:25-26 */
    MMIF_ST_SD = 1,     /* calc_std(f)    metric.py:30-34 */
    MMIF_ST_AG = 2,     /* calc_ag(f)     metric.py:38-46 */
    MMIF_ST_SF = 3,     /* calc_sf(f)     metric.py:50-59 */
    MMIF_ST_MSE_AF = 4, /* calc_mse(a,f)  metric.py:63-68 */
    MMIF_ST_MSE_BF = 5,
    MMIF_ST_CC_AF = 6,  /* calc_cc(a,f)   metric.py:80-91 */
    MMIF_ST_CC_BF = 7,
    MMIF_ST_SCD = 8,    /* calc_scd(a,b,f) metric.py:95-99 */
    MMIF_ST_MEAN_A = 9, MMIF_ST_MEAN_B = 10, MMIF_ST_SD_A = 11, MMIF_ST_SD_B = 12,
    MMIF_ST_CC_AB = 13,
    MMIF_ST_COUNT = 16
};
int mmif_stats(const float* a, const float* b, const float* f, int N, int H, int W, double* out,
               void* ws, size_t ws_bytes, void* stream);
/* Gradient of sum_c gout[c] * stat[c] over the MMIF_ST_* columns of the batch row `row` (device, MMIF_ST_COUNT
 * doubles: what mmif_stats returns for N = 1, the whole-batch combination for N > 1).  gout: device, MMIF_ST_COUNT
 * floats.  da / db / df: device, N*H*W floats each, any of them NULL (not computed, not written).
 * The batch is one population (global means, variances, covariances); the AG / SF forward differences stay inside a
 * sample.  Where the reference's autograd gives NaN so does this: a zero sd or a 0/0 correlation puts NaN on every pixel
 * of the images it involves, an AG stencil with equal pixels on its three pixels.  A column whose gout is exactly 0
 * contributes nothing.  Checks of mmif_stats plus MMIF_E_NULL for a null row / gout and MMIF_E_ALIGN for a row that is
 * not 8-byte or a gout / gradient that is not 4-byte aligned; all three outputs NULL launches nothing.  No allocation,
 * no synchronisation; one launch, counted under MMIF_CNT_METRIC. */
int mmif_stats_bwd(const float* a, const float* b, const float* f, int N, int H, int W, const double* row,
                   const float* gout, float* da, float* db, float* df, void* stream);

enum { /* mmif_hist entropy outputs, per pair */
    MMIF_EN_A = 0, MMIF_EN_B = 1, MMIF_EN_F = 2, /* calc_entropy      metric.py:119-125 (float32 arithmetic) */
    MMIF_JE_AF = 3, MMIF_JE_BF = 4,              /* calc_joint_ent    metric.py:148-154 (float64) */
    MMIF_CE_AF = 5, MMIF_CE_BF = 6,              /* calc_cross_ent    metric.py:158-165 (float32 arithmetic) */
    MMIF_MI_AF = 7, MMIF_MI_BF = 8,              /* calc_mul_info     metric.py:169-188, normalized=False */
    MMIF_NMI_AF = 9, MMIF_NMI_BF = 10,           /* calc_mul_info(normalized=True) */
    MMIF_EN_COUNT = 12
};
#define MMIF_HIST_WORDS (3 * 256 + 2 * 65536)
/* Replaces calc_prob/calc_joint_prob histogramming (torch.histc metric.py:113, np.histogram2d
 * metric.py:141-143) and the entropy family.  counts: per pair MMIF_HIST_WORDS uint32
 * [hist_a 256 | hist_b 256 | hist_f 256 | joint_af 256x256 (row = a bin) | joint_bf 256x256];
 * must be zero-filled by the caller.  ent: per pair MMIF_EN_COUNT doubles (may be NULL). */
int mmif_hist(const float* a, const float* b, const float* f, int N, int H, int W,
              uint32_t* counts, double* ent, void* ws, size_t ws_bytes, void* stream);

/* calc_Qabf(a,b,f,L,full=True) (metric.py:233-256) -> per pair 4 doubles:
 * qabf, nabf (modified), labf, nabf_unmodified (calc_Nabf(modified=False), metric.py:273). */
int mmif_qabf(const float* a, const float* b, const float* f, int N, int H, int W, float L,
              double* out, void* ws, size_t ws_bytes, void* stream);
/* The same plus the raw sums behind the four ratios -> per pair 9 doubles: qabf, nabf, labf, nabf_unmodified,
 * sum(Qaf wa + Qbf wb), sum(wa + wb), sum of the nabf terms, sum of the labf terms, sum of the unmodified-nabf terms.
 * calc_Qabf on a batch (N > 1) is the ratio of the sums over all pairs (metric.py:233-256 sums over every dimension). */
#define MMIF_QABF_RAW_DOUBLES 9
int mmif_qabf_raw(const float* a, const float* b, const float* f, int N, int H, int W, float L,
                  double* out, void* ws, size_t ws_bytes, void* stream);

/* Window-based fusion quality indices (definitions: oracle/quality_index.py): Piella & Heijmans' Q, Q_W, Q_E on every
 * 8x8 box window and Yang et al.'s Q_Y on the 11x11 metric SSIM windows (sigma 1.5, data range 255).  One launch reads
 * a, b, f once; the Sobel magnitudes of Q_E are formed on chip.  Per pair MMIF_QIDX_DOUBLES doubles: the four indices of
 * the pair, then the raw sums behind them, so that a batch (one population) is a ratio of sums over all pairs:
 *   Q = sum_term / box_windows;  Q_W = sum_cterm / sum_c (Q when sum_c == 0);
 *   Q_E = Q_W * (sum_cterm_e / sum_c_e, or sum_term_e / box_windows when sum_c_e == 0);  Q_Y = sum_term_y / qy_windows.
 * MMIF_E_NULL for a null image / out, MMIF_E_SHAPE unless N >= 1 and H, W >= 11, MMIF_E_ALIGN for an image pointer that
 * is not 4-byte or an out / ws that is not 8-byte aligned, MMIF_E_WORKSPACE for a null or short ws (size from
 * mmif_quality_index_workspace_bytes, which is 0 for a rejected shape; zero-filled once, left zeroed).
 * No allocation, no synchronisation; one launch, counted under MMIF_CNT_METRIC. */
enum {
    MMIF_QIDX_Q = 0, MMIF_QIDX_QW = 1, MMIF_QIDX_QE = 2, MMIF_QIDX_QY = 3,
    MMIF_QIDX_SUM_TERM = 4,       /* sum over box windows of lambda Q0(a,f) + (1 - lambda) Q0(b,f) */
    MMIF_QIDX_BOX_WINDOWS = 5,    /* (H-7)(W-7) */
    MMIF_QIDX_SUM_CTERM = 6,      /* sum of C * term, C = max(var a, var b) */
    MMIF_QIDX_SUM_C = 7,
    MMIF_QIDX_SUM_TERM_E = 8,     /* the same three on the Sobel magnitudes */
    MMIF_QIDX_SUM_CTERM_E = 9,
    MMIF_QIDX_SUM_C_E = 10,
    MMIF_QIDX_SUM_TERM_Y = 11,    /* sum over the SSIM windows of the Q_Y terms */
    MMIF_QIDX_QY_WINDOWS = 12     /* (H-10)(W-10) */
};
#define MMIF_QIDX_DOUBLES 13
size_t mmif_quality_index_workspace_bytes(int N, int H, int W);
int mmif_quality_index(const float* a, const float* b, const float* f, int N, int H, int W, double* out,
                       void* ws, size_t ws_bytes, void* stream);

/* calc_ssim(x,f,win,data_range,use_padding,full=True) (metric.py:316-364) for the two pairs
 * (a,f) and (b,f) -> per pair 4 doubles: ssim_af, cs_af, ssim_bf, cs_bf (global means). */
int mmif_ssim(const float* a, const float* b, const float* f, int N, int H, int W, int win_size,
              float data_range, int use_padding, double* out, void* ws, size_t ws_bytes, void* stream);

/* calc_msssim (metric.py:368-402) for (a,f) and (b,f) -> per pair 2 + 5*4 doubles:
 * msssim_af, msssim_bf, then per level ssim_af, cs_af, ssim_bf, cs_bf. */
#define MMIF_MSSSIM_DOUBLES 22
int mmif_msssim(const float* a, const float* b, const float* f, int N, int H, int W, int win_size,
                float data_range, double* out, void* ws, size_t ws_bytes, void* stream);

/* calc_vif + calc_viff (metric.py:406-491) -> per pair 2 + 4*6 doubles: viff(simple=False),
 * viff(simple=True), then per scale sum num1, den1, num2, den2, num_sel, den_sel. */
#define MMIF_VIFF_DOUBLES 26
int mmif_viff(const float* a, const float* b, const float* f, int N, int H, int W, double* out,
              void* ws, size_t ws_bytes, void* stream);

/* The 16-metric row of eval.py:29-75 for N pairs -> per pair 16 doubles in eval.py order:
 * sd ag sf mse psnr cc scd en ce mi qabf nabf labf ssim msssim viff. */
#define MMIF_EVAL_METRICS 16
int mmif_eval_suite(const float* a, const float* b, const float* f, int N, int H, int W,
                    double* out, void* ws, size_t ws_bytes, void* stream);

/* Host-buffer convenience used by the end-to-end benchmark and by CPU-tensor callers
 * (eval.py:198-206 leaves its tensors on the host): copies the three host images to the
 * device scratch `dev_scratch` (3*N*H*W floats), runs mmif_eval_suite and copies the row back.
 * Synchronises `stream` before returning. */
int mmif_eval_suite_host(const float* a_host, const float* b_host, const float* f_host, int N, int H,
                         int W, double* out_host, float* dev_scratch, double* dev_out,
                         void* ws, size_t ws_bytes, void* stream);

/* ---- uint8 ingest (SURVEY 8(f).3): eval.py:182-194 decodes 8-bit images with cv2 and widens them to float32 on the
 * host; these entries take the 8-bit pixels and widen on the device (4x less host->device traffic, identical results:
 * the widening is exact).  dev_scratch: 3*N*H*W floats (device).  The _host form copies from host memory into
 * dev_u8 (3 * roundup16(N*H*W) bytes, device), runs the suite, copies the rows back and synchronises `stream`. */
int mmif_widen_u8(const unsigned char* src, size_t n, float* dst, void* stream);
/* dst[i] = float32(src[i]) / 255 in IEEE float32 division: the `uint8 / 255` scaling the reference's datasets apply on the host
 * (data/dataset.py via torchvision to_tensor) done on the device, bit-identical, so training sources can be shipped as bytes. */
int mmif_widen_u8_unit(const unsigned char* src, size_t n, float* dst, void* stream);

/* ---- bfloat16 / float16 images (an autocast training step: the network's output is bfloat16, or float16 with a
 * GradScaler).  The loss kernels compute in float32; these two streaming entries sit around them.
 * mmif_widen: dst[i] = float32(src[i]), exact (float16 subnormals, +-inf and NaN as torch.Tensor.float() gives them);
 *   src: n elements of src_dtype (2-byte aligned), dst: n floats (4-byte aligned).
 * mmif_narrow: dst[i] = round-to-nearest-even of scale[0] * src[i] to dst_dtype (scale: one DEVICE float, or NULL for
 *   no multiply); the product is formed as the rescale of the single-pass backward forms it, so the result is that
 *   backward's float32 gradient .to(dtype) bit for bit, overflow to +-inf in float16 included.  src and scale 4-byte,
 *   dst 2-byte aligned.
 * Both: MMIF_E_NULL for a null src / dst, MMIF_E_MODE for a dtype other than BF16 / F16, MMIF_E_ALIGN for a misaligned
 * pointer; n == 0 launches nothing.  No synchronisation, no allocation.  Counted under MMIF_CNT_AUX. */
enum { MMIF_DTYPE_F32 = 0, MMIF_DTYPE_BF16 = 1, MMIF_DTYPE_F16 = 2 };
int mmif_widen(const void* src, int src_dtype, size_t n, float* dst, void* stream);
int mmif_narrow(const float* src, const float* scale, size_t n, int dst_dtype, void* dst, void* stream);

int mmif_eval_suite_u8(const unsigned char* a, const unsigned char* b, const unsigned char* f, int N, int H, int W,
                       double* out, float* dev_scratch, void* ws, size_t ws_bytes, void* stream);
int mmif_eval_suite_u8_host(const unsigned char* a_host, const unsigned char* b_host, const unsigned char* f_host,
                            int N, int H, int W, double* out_host, unsigned char* dev_u8, float* dev_scratch,
                            double* dev_out, void* ws, size_t ws_bytes, void* stream);

/* NormLoss (reference loss.py:361-385): out[0] = weight * mean(|x|) (MMIF_NORM_L1) or weight * mean(x^2) over the n
 * elements of x (device double); ws: mmif_norm_workspace_bytes() bytes, zero-initialised once, 8-byte aligned.
 * _bwd: gx[i] = gout1[0] * weight / n * sign(x[i]) (or 2 x[i]). */
size_t mmif_norm_workspace_bytes(void);
int mmif_norm_loss(const float* x, size_t n, int norm, float weight, double* out, void* ws, size_t ws_bytes, void* stream);
int mmif_norm_loss_bwd(const float* x, size_t n, int norm, float weight, const float* gout1, float* gx, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMIF_B200_H_ */
