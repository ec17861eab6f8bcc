// Small data-movement operators around the stencil kernels: the MS-SSIM level step of the loss
// (loss.py:147-153) and its adjoint, reflect padding (use_padding=True, loss.py:45-47) and its adjoint,
// the TVLoss backward (loss.py:347-358), and the widening / narrowing between the float32 the loss kernels
// compute in and the uint8 / bfloat16 / float16 images around them.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace mmif {

__global__ void __launch_bounds__(256) halve1_kernel(const float* __restrict__ src, float* __restrict__ dst, int H, int W, int Ho, int Wo) {
    const int n = blockIdx.z;
    const int j = blockIdx.x * 64 + (threadIdx.x & 63), i = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (i >= Ho || j >= Wo) return;
    const float* s = src + (size_t)n * H * W;
    const int r0 = 2 * i, r1 = (2 * i + 1 < H) ? 2 * i + 1 : H - 2;
    const int c0 = 2 * j, c1 = (2 * j + 1 < W) ? 2 * j + 1 : W - 2;
    const float v = ((__ldg(s + (size_t)r0 * W + c0) + __ldg(s + (size_t)r0 * W + c1)) + __ldg(s + (size_t)r1 * W + c0)) +
                    __ldg(s + (size_t)r1 * W + c1);
    dst[((size_t)n * Ho + i) * Wo + j] = v * 0.25f;
}

// g_src += adjoint(halve)(g_dst): every source pixel belongs to one 2x2 cell; with an odd size the
// reflected pad row/column H (W) is a second reader of row H-2 (column W-2).
__global__ void __launch_bounds__(256) halve1_bwd_kernel(const float* __restrict__ gd, float* __restrict__ gs, int H, int W, int Ho, int Wo) {
    const int n = blockIdx.z;
    const int c = blockIdx.x * 64 + (threadIdx.x & 63), r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= H || c >= W) return;
    const float* g = gd + (size_t)n * Ho * Wo;
    const bool er = (H & 1) && (r == H - 2), ec = (W & 1) && (c == W - 2);
    float v = __ldg(g + (size_t)(r >> 1) * Wo + (c >> 1));
    if (er) v += __ldg(g + (size_t)((H - 1) >> 1) * Wo + (c >> 1));
    if (ec) v += __ldg(g + (size_t)(r >> 1) * Wo + ((W - 1) >> 1));
    if (er && ec) v += __ldg(g + (size_t)((H - 1) >> 1) * Wo + ((W - 1) >> 1));
    gs[((size_t)n * H + r) * W + c] += 0.25f * v;
}

__device__ __forceinline__ int reflect_idx(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * n - 2 - i : i); }

__global__ void __launch_bounds__(256) reflect_pad_kernel(const float* __restrict__ src, float* __restrict__ dst, int H, int W, int pad) {
    const int n = blockIdx.z, Hp = H + 2 * pad, Wp = W + 2 * pad;
    const int c = blockIdx.x * 64 + (threadIdx.x & 63), r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= Hp || c >= Wp) return;
    dst[((size_t)n * Hp + r) * Wp + c] = __ldg(src + ((size_t)n * H + reflect_idx(r - pad, H)) * W + reflect_idx(c - pad, W));
}

// g_src = adjoint(reflect_pad)(g_dst): gather over the (up to 3 x 3) padded positions that read pixel (r, c).
__global__ void __launch_bounds__(256) reflect_pad_bwd_kernel(const float* __restrict__ gd, float* __restrict__ gs, int H, int W, int pad) {
    const int n = blockIdx.z, Hp = H + 2 * pad, Wp = W + 2 * pad;
    const int c = blockIdx.x * 64 + (threadIdx.x & 63), r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= H || c >= W) return;
    const float* g = gd + (size_t)n * Hp * Wp;
    int rs[3] = {r, -r, 2 * H - 2 - r}, cs[3] = {c, -c, 2 * W - 2 - c};     // unpadded coordinates of the readers
    float v = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int rr = rs[a];
        if (rr < -pad || rr >= H + pad || (a > 0 && rr == r)) continue;       // r == 0 / H-1 reflect onto themselves: count once
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const int cc = cs[b];
            if (cc < -pad || cc >= W + pad || (b > 0 && cc == c)) continue;
            v += __ldg(g + (size_t)(rr + pad) * Wp + (cc + pad));
        }
    }
    gs[((size_t)n * H + r) * W + c] = v;
}

__device__ __forceinline__ float nder(float d, int norm) { return norm == MMIF_NORM_L1 ? ((d > 0.f) ? 1.f : ((d < 0.f) ? -1.f : 0.f)) : 2.f * d; }

__global__ void __launch_bounds__(256) tv_bwd_kernel(const float* __restrict__ x, const float* __restrict__ gout, float* __restrict__ gx,
                                                     int H, int W, int norm, float kv, float kh) {
    const int n = blockIdx.z;
    const int c = blockIdx.x * 64 + (threadIdx.x & 63), r = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (r >= H || c >= W) return;
    const float* p = x + (size_t)n * H * W;
    const float g = __ldg(gout), v = __ldg(p + (size_t)r * W + c);
    float acc = 0.f;
    if (r > 0) acc += kv * nder(v - __ldg(p + (size_t)(r - 1) * W + c), norm);
    if (r + 1 < H) acc -= kv * nder(__ldg(p + (size_t)(r + 1) * W + c) - v, norm);
    if (c > 0) acc += kh * nder(v - __ldg(p + (size_t)r * W + c - 1), norm);
    if (c + 1 < W) acc -= kh * nder(__ldg(p + (size_t)r * W + c + 1) - v, norm);
    gx[((size_t)n * H + r) * W + c] = g * acc;
}

// ---- Widening to float32, exact for every source type below.
// uint8 ingest (eval.py:182-194 decodes 8-bit images and widens them on the host; widening on the device cuts the
// host->device traffic of an evaluation 4x).  U8Unit divides by 255 in IEEE float32 division — bit-identical to the
// `uint8 -> float32 / 255` of the reference's input pipeline (data/dataset.py through torchvision's to_tensor), so a
// training loop can ship 8-bit sources to the device.
// bfloat16 / float16 images of an autocast training step enter the float32 loss kernels the same way: the value is
// what torch.Tensor.float() gives (float16 subnormals, +-inf and NaN included).
// Each source type names its storage bits and the float32 value of one element's bits.
struct SrcU8 {
    using bits = unsigned char;
    static __device__ __forceinline__ float widen1(unsigned v) { return (float)v; }
};
struct SrcU8Unit {
    using bits = unsigned char;
    static __device__ __forceinline__ float widen1(unsigned v) { return __fdiv_rn((float)v, 255.0f); }
};
struct SrcBF16 {
    using bits = unsigned short;
    static __device__ __forceinline__ float widen1(unsigned v) { return __uint_as_float(v << 16); }
};
struct SrcF16 {
    using bits = unsigned short;
    static __device__ __forceinline__ float widen1(unsigned v) { return __half2float(__ushort_as_half((unsigned short)v)); }
};

// One 16-byte load per thread and iteration (16 uint8 or 8 half-width elements), float4 stores; vec = both pointers 16-byte
// aligned, else element by element.
template <typename S>
__global__ void __launch_bounds__(256) widen_kernel(const typename S::bits* __restrict__ src, float* __restrict__ dst, size_t n, int vec) {
    constexpr int kBits = 8 * (int)sizeof(typename S::bits), kPer = 128 / kBits;
    constexpr unsigned kMask = (1u << kBits) - 1u;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec) {
        const size_t nv = n / kPer;
        const uint4* s16 = reinterpret_cast<const uint4*>(src);
        float4* d4 = reinterpret_cast<float4*>(dst);
        for (; i < nv; i += stride) {
            const uint4 v = __ldg(s16 + i);
            const unsigned w[4] = {v.x, v.y, v.z, v.w};
            float e[kPer];
#pragma unroll
            for (int k = 0; k < kPer; ++k) e[k] = S::widen1((w[k * kBits / 32] >> (k * kBits % 32)) & kMask);
#pragma unroll
            for (int k = 0; k < kPer / 4; ++k) d4[(kPer / 4) * i + k] = make_float4(e[4 * k], e[4 * k + 1], e[4 * k + 2], e[4 * k + 3]);
        }
        for (size_t t = nv * kPer + (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) dst[t] = S::widen1(src[t]);
    } else {
        for (; i < n; i += stride) dst[i] = S::widen1(src[i]);
    }
}

// ---- Narrowing of a float32 gradient to the bfloat16 / float16 of the image it belongs to: dst = RNE(scale[0] * src), the
// product formed as rescale_unit_kernel forms it (g0 * v), so the result is that kernel's float32 gradient .to(dtype) bit
// for bit, overflow to +-inf in float16 included (what a GradScaler detects).  scale == NULL: dst = RNE(src).
template <typename D> __device__ __forceinline__ D narrow1(float v);
template <> __device__ __forceinline__ __nv_bfloat16 narrow1<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half narrow1<__half>(float v) { return __float2half_rn(v); }

// vec = src 16-byte and dst 8-byte aligned: one float4 load and one 8-byte store per thread and iteration.
template <typename D>
__global__ void __launch_bounds__(256) narrow_kernel(const float* __restrict__ src, const float* __restrict__ scale, D* __restrict__ dst,
                                                     size_t n, int vec) {
    const bool scaled = scale != nullptr;
    const float g0 = scaled ? __ldg(scale) : 1.f;
    auto one = [&](float v) { return narrow1<D>(scaled ? g0 * v : v); };
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec) {
        const size_t n4 = n >> 2;
        const float4* s4 = reinterpret_cast<const float4*>(src);
        uint2* d4 = reinterpret_cast<uint2*>(dst);
        for (; i < n4; i += stride) {
            const float4 v = __ldcs(s4 + i);
            const D o[4] = {one(v.x), one(v.y), one(v.z), one(v.w)};
            uint2 u;
            memcpy(&u, o, sizeof(u));
            d4[i] = u;
        }
        for (size_t t = (n4 << 2) + (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) dst[t] = one(src[t]);
    } else {
        for (; i < n; i += stride) dst[i] = one(src[i]);
    }
}

// ---- NormLoss (loss.py:361-385): weight * mean(|x|) or weight * mean(x^2) of an arbitrary tensor, and its gradient.
// Deterministic: per-CTA partials in double, the last CTA to arrive adds them in index order.
constexpr int kNormBlocks = 592;
__global__ void __launch_bounds__(256) norm_loss_kernel(const float* __restrict__ x, size_t n, int norm, double scale, unsigned* counter,
                                                        double* partial, double* out) {
    __shared__ double red[8];
    __shared__ int flag;
    float acc = 0.f;
    double total = 0.0;
    int cnt = 0;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        const float v = __ldg(x + i);
        acc += (norm == MMIF_NORM_L1) ? fabsf(v) : v * v;
        if (++cnt == 64) { total += (double)acc; acc = 0.f; cnt = 0; }       // bound the float run length
    }
    double v1[1] = {total + (double)acc};
    block_sum<1, 256>(v1, red);
    if (threadIdx.x == 0) {
        partial[blockIdx.x] = v1[0];
        __threadfence();
        flag = (atomicAdd(counter, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!flag) return;
    __threadfence();
    double t[1] = {0.0};
    for (int k = threadIdx.x; k < (int)gridDim.x; k += 256) t[0] += __ldcg(partial + k);
    block_sum<1, 256>(t, red);
    if (threadIdx.x == 0) { out[0] = t[0] * scale; *counter = 0u; }
}
__global__ void __launch_bounds__(256) norm_loss_bwd_kernel(const float* __restrict__ x, size_t n, int norm, float k, const float* __restrict__ gout,
                                                            float* __restrict__ gx) {
    const float g = __ldg(gout) * k;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        const float v = __ldg(x + i);
        gx[i] = g * ((norm == MMIF_NORM_L1) ? ((v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f)) : 2.f * v);
    }
}

static int chk(const void* a, const void* b, int N, int H, int W) {
    if (!a || !b) { set_error("null pointer"); return MMIF_E_NULL; }
    if (N < 1 || H < 2 || W < 2) { set_error("bad shape (%d,%d,%d)", N, H, W); return MMIF_E_SHAPE; }
    if (((uintptr_t)a | (uintptr_t)b) & 3) { set_error("pointers must be 4-byte aligned"); return MMIF_E_ALIGN; }
    return MMIF_OK;
}

}  // namespace mmif

using namespace mmif;

extern "C" int mmif_halve(const float* src, int N, int H, int W, float* dst, void* stream) {
    int rc = chk(src, dst, N, H, W); if (rc) return rc;
    const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
    halve1_kernel<<<dim3(ceil_div(Wo, 64), ceil_div(Ho, 4), N), 256, 0, (cudaStream_t)stream>>>(src, dst, H, W, Ho, Wo);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
extern "C" int mmif_halve_bwd(const float* g_dst, int N, int H, int W, float* g_src_accum, void* stream) {
    int rc = chk(g_dst, g_src_accum, N, H, W); if (rc) return rc;
    const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
    halve1_bwd_kernel<<<dim3(ceil_div(W, 64), ceil_div(H, 4), N), 256, 0, (cudaStream_t)stream>>>(g_dst, g_src_accum, H, W, Ho, Wo);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
extern "C" int mmif_reflect_pad(const float* src, int N, int H, int W, int pad, float* dst, void* stream) {
    int rc = chk(src, dst, N, H, W); if (rc) return rc;
    if (pad < 0 || pad >= H || pad >= W) { set_error("reflect pad %d must be smaller than H, W", pad); return MMIF_E_SHAPE; }
    reflect_pad_kernel<<<dim3(ceil_div(W + 2 * pad, 64), ceil_div(H + 2 * pad, 4), N), 256, 0, (cudaStream_t)stream>>>(src, dst, H, W, pad);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
extern "C" int mmif_reflect_pad_bwd(const float* g_dst, int N, int H, int W, int pad, float* g_src, void* stream) {
    int rc = chk(g_dst, g_src, N, H, W); if (rc) return rc;
    if (pad < 0 || pad >= H || pad >= W) { set_error("reflect pad %d must be smaller than H, W", pad); return MMIF_E_SHAPE; }
    reflect_pad_bwd_kernel<<<dim3(ceil_div(W, 64), ceil_div(H, 4), N), 256, 0, (cudaStream_t)stream>>>(g_dst, g_src, H, W, pad);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
extern "C" int mmif_tv_loss_bwd(const float* x, int N, int H, int W, int norm, float weight, const float* gout1, float* gx,
                                void* stream) {
    int rc = chk(x, gx, N, H, W); if (rc) return rc;
    if (!gout1) { set_error("null gout1"); return MMIF_E_NULL; }
    if (norm != MMIF_NORM_L1 && norm != MMIF_NORM_L2) { set_error("unsupported norm"); return MMIF_E_MODE; }
    const float kv = weight / ((float)N * (float)(H - 1) * (float)W), kh = weight / ((float)N * (float)H * (float)(W - 1));
    tv_bwd_kernel<<<dim3(ceil_div(W, 64), ceil_div(H, 4), N), 256, 0, (cudaStream_t)stream>>>(x, gout1, gx, H, W, norm, kv, kh);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}

// grid of the streaming kernels: one 16-byte source load per thread, at most 16 CTAs per SM (grid-stride beyond that)
static unsigned stream_blocks(size_t n, size_t per_thread) {
    const size_t blocks = (n / per_thread + 255) / 256;
    return (unsigned)(blocks < 1 ? 1 : (blocks > 148 * 16 ? 148 * 16 : blocks));
}
template <typename S>
static int widen_launch(const void* src, size_t n, float* dst, void* stream) {
    const int vec = ((((uintptr_t)src) | ((uintptr_t)dst)) & 15) == 0;
    widen_kernel<S><<<stream_blocks(n, 16 / sizeof(typename S::bits)), 256, 0, (cudaStream_t)stream>>>(
        (const typename S::bits*)src, dst, n, vec);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
static int widen_impl(const unsigned char* src, size_t n, float* dst, void* stream, bool unit);
extern "C" int mmif_widen_u8(const unsigned char* src, size_t n, float* dst, void* stream) { return widen_impl(src, n, dst, stream, false); }
extern "C" int mmif_widen_u8_unit(const unsigned char* src, size_t n, float* dst, void* stream) { return widen_impl(src, n, dst, stream, true); }
static int widen_impl(const unsigned char* src, size_t n, float* dst, void* stream, bool unit) {
    if (!src || !dst) { set_error("null pointer"); return MMIF_E_NULL; }
    if (((uintptr_t)dst) & 3) { set_error("dst must be 4-byte aligned"); return MMIF_E_ALIGN; }
    if (n == 0) return MMIF_OK;
    return unit ? widen_launch<SrcU8Unit>(src, n, dst, stream) : widen_launch<SrcU8>(src, n, dst, stream);
}
extern "C" int mmif_widen(const void* src, int src_dtype, size_t n, float* dst, void* stream) {
    if (!src || !dst) { set_error("null pointer"); return MMIF_E_NULL; }
    if (src_dtype != MMIF_DTYPE_BF16 && src_dtype != MMIF_DTYPE_F16) { set_error("widen: source dtype %d is not BF16 / F16", src_dtype); return MMIF_E_MODE; }
    if ((((uintptr_t)src) & 1) || (((uintptr_t)dst) & 3)) { set_error("widen: src must be 2-byte, dst 4-byte aligned"); return MMIF_E_ALIGN; }
    if (n == 0) return MMIF_OK;
    return src_dtype == MMIF_DTYPE_BF16 ? widen_launch<SrcBF16>(src, n, dst, stream) : widen_launch<SrcF16>(src, n, dst, stream);
}
extern "C" int mmif_narrow(const float* src, const float* scale, size_t n, int dst_dtype, void* dst, void* stream) {
    if (!src || !dst) { set_error("null pointer"); return MMIF_E_NULL; }
    if (dst_dtype != MMIF_DTYPE_BF16 && dst_dtype != MMIF_DTYPE_F16) { set_error("narrow: destination dtype %d is not BF16 / F16", dst_dtype); return MMIF_E_MODE; }
    if (((((uintptr_t)src) | ((uintptr_t)scale)) & 3) || (((uintptr_t)dst) & 1)) {
        set_error("narrow: src and scale must be 4-byte, dst 2-byte aligned");
        return MMIF_E_ALIGN;
    }
    if (n == 0) return MMIF_OK;
    const int vec = (((uintptr_t)src) & 15) == 0 && (((uintptr_t)dst) & 7) == 0;
    const unsigned blocks = stream_blocks(n, 4);
    if (dst_dtype == MMIF_DTYPE_BF16)
        narrow_kernel<__nv_bfloat16><<<blocks, 256, 0, (cudaStream_t)stream>>>(src, scale, (__nv_bfloat16*)dst, n, vec);
    else
        narrow_kernel<__half><<<blocks, 256, 0, (cudaStream_t)stream>>>(src, scale, (__half*)dst, n, vec);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
extern "C" size_t mmif_norm_workspace_bytes(void) { return 256 + (size_t)kNormBlocks * sizeof(double); }
extern "C" int mmif_norm_loss(const float* x, size_t n, int norm, float weight, double* out, void* ws, size_t ws_bytes, void* stream) {
    if (!x || !out || !ws) { set_error("null pointer"); return MMIF_E_NULL; }
    if (n == 0) { set_error("empty tensor"); return MMIF_E_SHAPE; }
    if (norm != MMIF_NORM_L1 && norm != MMIF_NORM_L2) { set_error("unsupported norm"); return MMIF_E_MODE; }
    if (ws_bytes < mmif_norm_workspace_bytes() || (((uintptr_t)ws) & 7)) { set_error("norm workspace too small / unaligned"); return MMIF_E_WORKSPACE; }
    size_t blocks = (n + 2047) / 2048;
    blocks = blocks < 1 ? 1 : (blocks > (size_t)kNormBlocks ? (size_t)kNormBlocks : blocks);
    norm_loss_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, norm, (double)weight / (double)n, (unsigned*)ws,
                                                                          (double*)((unsigned char*)ws + 256), out);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
extern "C" int mmif_norm_loss_bwd(const float* x, size_t n, int norm, float weight, const float* gout1, float* gx, void* stream) {
    if (!x || !gout1 || !gx) { set_error("null pointer"); return MMIF_E_NULL; }
    if (norm != MMIF_NORM_L1 && norm != MMIF_NORM_L2) { set_error("unsupported norm"); return MMIF_E_MODE; }
    if (n == 0) return MMIF_OK;
    size_t blocks = (n + 1023) / 1024;
    blocks = blocks > 148 * 16 ? 148 * 16 : blocks;
    norm_loss_bwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, norm, weight / (float)n, gout1, gx);
    mmif::count_launch(MMIF_CNT_AUX);
    MMIF_CUDA(cudaGetLastError());
    return MMIF_OK;
}
