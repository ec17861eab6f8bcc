// Warp-specialised form of the loss + gradient kernel (included by fusion_loss.cu; same arithmetic, same tile geometry,
// bit-identical gradients for equal row segments).
//
// Why: fusion_loss_bwd_kernel keeps all five phases of a batch in every thread, needs 255 registers for that and so runs
// 2 CTAs x 4 warps per SM = TWO warps per scheduler; ncu (profiles/r2_zkernel.txt) shows the FP32 pipe 65 % busy with
// the schedulers idle on `wait` / `short_scoreboard` / `no_instruction` / `barrier`: too few warps to cover each other.
// Here ONE CTA of 512 threads owns the SM and its four warp groups are pipeline stages working on different batches
// at the same time, handing the tile on through shared memory (no CTA-wide barrier in the batch loop):
//   G0 (warps 0-3)   : TMA producer + vertical moments V(b): ring -> vbuf[b & 1]
//   G1 (warps 4-7)   : horizontal moments + SSIM derivative coefficients H(b): vbuf[b & 1] -> cbuf[b & 1]
//   G2 (warps 8-11)  : Sobel / pixel adjoint S(b): ring -> gbuf[b & 1]
//   G3 (warps 12-15) : vertical adjoint B1(b) (stateful) cbuf -> tbuf, horizontal adjoint + combine + store B2(b)
// Each group keeps only its own phase's registers (<= 128), every scheduler holds four warps of four different phases
// (FMA-heavy blur next to the issue-bound Sobel / epilogue code), and a stage never waits for the whole CTA.
// What the captures taught (profiles/r2b_ws_steps.txt), in the order it was learnt:
//   * three or four instruction streams per SM thrash the 32 KB L1.5 instruction cache if the fully unrolled bodies
//     (43 KB) are kept: `no_instruction` went from 0.27 to 2.33 stalls per issue.  H, S are therefore two passes over half
//     the tile through ONE copy of the code (B1 / B2 / V stay unrolled: the total is ~30 KB) -> 0.2;
//   * mbarrier try_wait / nanosleep polling by the waiting groups executed 40 % of all instructions; the SM's dispatch
//     port turned out to be the binding resource (a packed FFMA2 holds it for two cycles: issue 62 % + packed shadows 30 %
//     = 92-94 % busy), so the hand-overs between groups are HARDWARE named barriers (bar.arrive / bar.sync: a blocked warp
//     issues nothing) and only the TMA ring keeps mbarriers;
//   * with the port saturated the only remaining lever is the instruction count per batch (~2.6 k per 8 x 128 tile now).
// Shared memory (213 KB of the SM's 227): 7-slot input ring (G3's combine reads rows three batches behind G0's prefetch),
// double-buffered vbuf / cbuf / gbuf, one tbuf.
#pragma once

namespace mmif {

constexpr int kWsSlots = 7;
constexpr int kWsRows = kWsSlots * kRB;     // 56 ring rows
constexpr int kWsNT = 512;
#ifndef MMIF_WS_SLEEP_NS
#define MMIF_WS_SLEEP_NS 40
#endif
constexpr unsigned kWsSleepNs = MMIF_WS_SLEEP_NS;
#ifndef MMIF_WS_NO_SFAST
#define MMIF_WS_NO_SFAST 0
#endif
#ifndef MMIF_WS_H_UNROLL
#define MMIF_WS_H_UNROLL 0
#endif
constexpr int kWsGroupBytes = 3 * kRB * kRPB * 4;

struct SmemWS {
    float ring[3][kWsRows][kRPB];                      // 88704 B
    alignas(16) float2 vbuf[2][kRB * kVPitch];         // 2 x 34944 B
    alignas(16) float2 cbuf[2][kRB * kCPitch];         // 2 x 16512 B
    alignas(16) float2 tbuf[kRB * kCPitch];            // 16512 B
    alignas(16) float gbuf[2][kRB][kTMC + 4];          // 2 x 4224 B
    unsigned long long ring_full[kWsSlots], ring_empty[kWsSlots];
    double red[8 * (kWsNT / 32)];
    float shift_scratch[(kWsNT / 32) * 3];
    int flag;
};

// One arrival per WARP (lane 0, after the warp's lanes have synchronised their shared-memory accesses): the barriers count
// warps, not threads.  With 128 arrivals per phase every arrival woke the sleeping waiters, and their re-checks were
// 20 % of all executed instructions (ncu source page).
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Every thread arrives (the plain-load ring: each thread publishes its own stores; also what compute-sanitizer's racecheck
// can follow).
__device__ __forceinline__ void mbar_arrive_each(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Poll with a real sleep between the tests and a watchdog (a protocol error traps: the launch fails instead of hanging the
// GPU).  Only the TMA ring is waited on this way; try_wait's own suspend returned after ~100 cycles and the polling loops of
// the first version executed 40 % of all instructions, hence named barriers everywhere else.
__device__ __forceinline__ void mbar_wait_wd(unsigned long long* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t ok = 0;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
    for (unsigned spin = 0; !ok; ++spin) {
        __nanosleep(kWsSleepNs);           // a real sleep between polls: try_wait's own suspend returns after a few cycles
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(addr), "r"(parity)
            : "memory");
        if (spin > (1u << 24)) __trap();
    }
}
__device__ __forceinline__ void group_sync(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }
// Producer / consumer hand-over between two warp groups on a HARDWARE named barrier (256 = the 128 arriving + the 128 waiting
// threads): a warp blocked in bar.sync issues nothing, whereas the mbarrier polling loops of the first version of this kernel
// executed 40 % of all instructions (ncu source page) on a dispatch port that is the kernel's bottleneck.  Every barrier has
// at most one phase in flight (full / empty pairs over double buffers).
enum { NB_TBUF = 1, NB_VFULL = 2, NB_VEMPTY = 4, NB_CFULL = 6, NB_CEMPTY = 8, NB_GFULL = 10, NB_GEMPTY = 12 };
__device__ __forceinline__ void nb_sync(int id) { asm volatile("bar.sync %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id) { asm volatile("bar.arrive %0, 256;" ::"r"(id) : "memory"); }
__device__ __forceinline__ int ws_wrap(int r) { return r >= kWsRows ? r - kWsRows : r; }      // r in [0, 2 kWsRows)

// tile_shift of stencil.cuh for the 384-thread CTA: every warp group samples the same 16 x 8 grid, so all threads end up
// with the same constants (and the same ones as the 128-thread kernels).
__device__ __forceinline__ Shift tile_shift_ws(float* scratch, const float* x1, const float* x2, const float* y, int H, int W, int r0,
                                               int nr, int c0, const Taps& tp) {
    const int tl = threadIdx.x & 127;
    int r = r0 + ((tl >> 4) * nr) / 8 + nr / 16;
    int c = c0 + (tl & 15) * 8 + 4;
    r = min(max(r, 0), H - 1);
    c = min(max(c, 0), W - 1);
    const size_t off = (size_t)r * W + c;
    float v[3] = {__ldg(x1 + off), __ldg(x2 + off), __ldg(y + off)};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (!(fabsf(v[k]) <= 3.0e38f)) v[k] = 3.0e38f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] = fminf(v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
    }
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { scratch[warp * 3 + 0] = v[0]; scratch[warp * 3 + 1] = v[1]; scratch[warp * 3 + 2] = v[2]; }
    __syncthreads();
    float c3[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float m = scratch[k];
#pragma unroll
        for (int w = 1; w < 4; ++w) m = fminf(m, scratch[w * 3 + k]);
        c3[k] = (m < 3.0e38f) ? m : 0.f;
    }
    __syncthreads();
    return make_shift(c3[0], c3[1], c3[2], tp.wsum, tp.weps, tp.wrho);
}

// ZMODE: 0 = gradient only, 1 = gradient + all loss sums (per-sample ssim / cs / sigma means, pixel, grad), 2 = gradient + the sums
// the training objective consumes (ssim, pixel, grad; the cs / sigma entries of the per-sample block are written as 0).
template <int WIN, bool FAST, int ZMODE>
__global__ void __launch_bounds__(kWsNT, 1)
fusion_loss_ws_kernel(const __grid_constant__ CUtensorMap map1, const __grid_constant__ CUtensorMap map2,
                      const __grid_constant__ CUtensorMap mapy, const BwdParams p) {
    constexpr int HALO = BG<WIN>::HALO, kOFF = BG<WIN>::OFF, kVOFF = BG<WIN>::VOFF, kTG = BG<WIN>::TG, kWC = BG<WIN>::WC;
    const bool unit_up = (p.gout[0] == nullptr) && (p.gout[1] == nullptr) && (p.gout[2] == nullptr);
    const float g_ssim = unit_up ? 1.f : (p.gout[0] ? __ldg(p.gout[0]) : 0.f);
    const float g_pix = unit_up ? 1.f : (p.gout[1] ? __ldg(p.gout[1]) : 0.f);
    const float g_grad = unit_up ? 1.f : (p.gout[2] ? __ldg(p.gout[2]) : 0.f);
    if (!ZMODE && p.dF_unit != nullptr && g_ssim == g_pix && g_pix == g_grad) return;     // rescale_unit_kernel did the work
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SmemWS& sm = *reinterpret_cast<SmemWS*>(smem_raw);
    // Linear CTA index -> (class, segment, sample, strip).  Dispatch order = launch order: all tall segments of the coarse
    // strips, then their short segments, then the fine class (the last fine_strips strips of every sample in segments of
    // fine_rows rows): longest jobs first, the fine ones level the SMs at the end.
    const int sa = p.nstrip - p.fine_strips;              // coarse strips per sample
    const int cols_a = p.B * sa, n_a = cols_a * p.nseg;
    int id = blockIdx.x, seg, strip, n, i0, seg_h, blk;
    if (id < n_a) {
        seg = id / cols_a;
        const int lin = id - seg * cols_a;
        n = lin / sa;
        strip = lin - n * sa;
        i0 = (seg < p.n_tall) ? seg * p.seg_rows : p.n_tall * p.seg_rows + (seg - p.n_tall) * p.seg_short;
        seg_h = (seg < p.n_tall) ? p.seg_rows : p.seg_short;
        blk = seg * sa + strip;
    } else {
        id -= n_a;
        const int cols_f = p.B * p.fine_strips;
        seg = id / cols_f;
        const int lin = id - seg * cols_f;
        n = lin / p.fine_strips;
        strip = sa + (lin - n * p.fine_strips);
        i0 = seg * p.fine_rows;
        seg_h = p.fine_rows;
        blk = sa * p.nseg + seg * p.fine_strips + (strip - sa);
    }
    const int nblk = sa * p.nseg + p.fine_strips * p.nseg_fine;
    const int j0 = strip * kTG;
    const int jw0 = j0 - kOFF;
    const int R0 = i0 - HALO;
    const int iend = min(i0 + seg_h, p.H);
    const int jend = min(j0 + kTG, p.W);
    const int nb = (iend - R0 + kRB - 1) / kRB;
    const size_t img_off = (size_t)n * p.H * p.W;
    const int grp = threadIdx.x >> 7;
    const int t = threadIdx.x & 127;              // index within the warp group
    const int lane = t & 31, warp = t >> 5;
    const bool use_tma = p.use_tma != 0;
    const float* img[3] = {p.x1 + img_off, p.x2 + img_off, p.y + img_off};

    if (threadIdx.x == 0) {
        for (int s = 0; s < kWsSlots; ++s) {
            mbar_init((uint64_t*)&sm.ring_full[s], use_tma ? 1 : 128);
            mbar_init((uint64_t*)&sm.ring_empty[s], 8);         // warps of G2 (after S) + G3 (after B2)
        }
        mbar_fence_init();
    }
    __syncthreads();
    // the first three ring groups are requested BEFORE the tile shift is sampled (two CTA barriers and a dependent global load):
    // their latency is the longest item of a short CTA's prologue
    auto issue = [&](int g) {               // input rows R0 + 8 g .. + 8 of the three images -> ring slot g % kWsSlots
        const int slot = g % kWsSlots;
        const uint32_t par = ((g / kWsSlots) & 1) ^ 1;
        if (use_tma) {
            if (t == 0) {
                mbar_wait_wd(&sm.ring_empty[slot], par);
                uint64_t* bar = (uint64_t*)&sm.ring_full[slot];
                mbar_expect_tx(bar, kWsGroupBytes);
                tma_load_3d(&sm.ring[0][slot * kRB][0], &map1, jw0, R0 + g * kRB, n, bar);
                tma_load_3d(&sm.ring[1][slot * kRB][0], &map2, jw0, R0 + g * kRB, n, bar);
                tma_load_3d(&sm.ring[2][slot * kRB][0], &mapy, jw0, R0 + g * kRB, n, bar);
            }
        } else {
            mbar_wait_wd(&sm.ring_empty[slot], par);
            for (int tc = t; tc < kRPB; tc += 128) {
                const int col = jw0 + tc;
                const bool cok = (col >= 0) && (col < p.W);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
#pragma unroll
                    for (int r = 0; r < kRB; ++r) {
                        const int row = R0 + g * kRB + r;
                        float v = 0.f;
                        if (cok && row >= 0 && row < p.H) v = __ldg(img[k] + (size_t)row * p.W + col);
                        sm.ring[k][slot * kRB + r][tc] = v;
                    }
                }
            }
            mbar_arrive_each(&sm.ring_full[slot]);
        }
    };
    if (grp == 0) {
        issue(0);
        issue(1);
        issue(2);
    }
    const Shift sh = tile_shift_ws(sm.shift_scratch, img[0], img[1], img[2], p.H, p.W, R0, iend - R0 + HALO, jw0, p.taps);
    double zv[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};

    if (grp == 0) {
        // =========================================================== G0: input ring (TMA producer), vertical moments
        // Scatter form: each input row is loaded, shifted and multiplied ONCE and FMA'd into the WIN window rows it belongs
        // to; the HALO window rows still open at the end of a batch are carried into the next one (a gather over the 18
        // input rows of a batch would redo the loads and products of 10 of them).  Every window row still receives its
        // taps in the order 0 .. WIN - 1, tap 0 as a multiply, so the sums are bit-identical to the gather form's.
        static_assert(HALO <= 2 * kRB, "a batch's input rows must lie in three ring slots");
        float2 acc[kRB + HALO][4];                      // window rows Rb .. Rb + 17 of batch b; [0, HALO) carried in
        const float2 negc = f2(-sh.c.x, -sh.c.y);
        // input row rr of the batch (ring row rp) -> tap rr - o of every open window row o <= rr
        auto vrow = [&](const float* rp, const int rr) {
            const float y = rp[2 * kWsRows * kRPB] - sh.cy;
            float2 P[4];
            P[0] = add2(f2(rp[0], rp[kWsRows * kRPB]), negc);
            P[1] = mul2(P[0], P[0]);
            P[2] = muls(y, P[0]);
            P[3] = f2(y, y * y);
            // window rows in ascending order (taps descending): then the last row of a batch finishes window row o before
            // it writes row o + kRB, whose value is carried in the registers of row o, and the carry needs no moves
#pragma unroll
            for (int k = WIN - 1; k >= 0; --k) {
                const int o = rr - k;
                if (o >= 0) {
#pragma unroll
                    for (int m = 0; m < 4; ++m) acc[o][m] = (k == 0) ? muls(p.taps.w[0], P[m]) : fmas(p.taps.w[k], P[m], acc[o][m]);
                }
            }
        };
        mbar_wait_wd(&sm.ring_full[0], 0);
        mbar_wait_wd(&sm.ring_full[1], 0);
        {   // warm-up: input rows R0 .. R0 + HALO - 1 (ring slots 0 and 1) open window rows 0 .. HALO - 1 of batch 0
            const float* q0 = &sm.ring[0][0][t + kVOFF];
#pragma unroll
            for (int rr = 0; rr < HALO; ++rr) vrow(q0 + rr * kRPB, rr);
        }

        int slot = 0;                                   // b % kWsSlots
        for (int b = 0; b < nb; ++b) {
            if (b + 1 < nb) issue(b + 3);
            mbar_wait_wd(&sm.ring_full[(slot + 2) % kWsSlots], ((b + 2) / kWsSlots) & 1);
            // ---- V(b): vertical moments of window rows [Rb, Rb+8) -> vbuf[b & 1]
            if (b >= 2) nb_sync(NB_VEMPTY + (b & 1));             // H(b - 2) has read this vbuf
            {
                // the batch's new input rows Rb + HALO .. Rb + HALO + 7 lie in the next two ring slots: two base pointers,
                // constant row offsets, no per-row wrap arithmetic
                float2* vb = sm.vbuf[b & 1];
                const int s1 = (slot + 1 == kWsSlots) ? 0 : slot + 1, s2 = (s1 + 1 == kWsSlots) ? 0 : s1 + 1;
                const float* sg[3] = {nullptr, &sm.ring[0][s1 * kRB][t + kVOFF], &sm.ring[0][s2 * kRB][t + kVOFF]};
#pragma unroll
                for (int rr = HALO; rr < kRB + HALO; ++rr) {
                    vrow(sg[rr >> 3] + (rr & 7) * kRPB, rr);
                    const int o = rr - HALO;                    // window row o has all its taps
#pragma unroll
                    for (int m = 0; m < 4; ++m) vb[o * kVPitch + m * kVCols + t] = acc[o][m];
                }
#pragma unroll
                for (int d = 0; d < HALO; ++d) {
#pragma unroll
                    for (int m = 0; m < 4; ++m) acc[d][m] = acc[d + kRB][m];
                }
            }
            nb_arrive(NB_VFULL + (b & 1));
            slot = (slot + 1 == kWsSlots) ? 0 : slot + 1;
        }
    } else if (grp == 1) {
        // =========================================================== G1: horizontal moments -> derivative coefficients
        const int ho = lane & 7, hg = warp * 4 + (lane >> 3);
        float2 z_ss = f2(0.f, 0.f), z_cs = z_ss, z_sg = z_ss;
        // bit j: the SSIM value of window column hg * 8 + j belongs to this CTA's tile (single-pass loss sums).  Window columns
        // that do not exist (outside the image) need no mask here: G3 zeroes their vertical-adjoint output, and the columns
        // past the strip's 118 are never read by the horizontal adjoint.
        unsigned a_zmask = 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int pw = hg * 8 + j, pc = jw0 + kVOFF + pw;
            const bool v = (pw < kWC) && (pc >= 0) && (pc < p.Wout);
            a_zmask |= (v && pc >= j0 && pc < jend) ? (1u << j) : 0u;
        }
        for (int b = 0; b < nb; ++b) {
            const int Rb = R0 + b * kRB;
            const int q = Rb + ho;
            const bool active = (hg * 8 < kWC) && (q >= 0) && (q < p.Hout);
            nb_sync(NB_VFULL + (b & 1));
            if (b >= 2) nb_sync(NB_CEMPTY + (b & 1));             // B1(b - 2) has read this cbuf
            const unsigned zm = (ZMODE && q >= i0 && q < iend) ? a_zmask : 0u;
            // two passes of four window columns through ONE copy of the code: the instruction footprint of the three
            // concurrent streams has to fit the SM's 32 KB instruction cache
#if MMIF_WS_H_UNROLL
#pragma unroll
#else
#pragma unroll 1
#endif
            for (int half = 0; half < 2; ++half) {
                float2 ab[4], cc[4];
                const unsigned zmh = zm >> (half * 4);
                if (active) {
                    float2 acc[4][4];
                    hpass<WIN, 4, false, 4>(sm.vbuf[b & 1] + ho * kVPitch + hg * 8 + half * 4, kVCols, p.taps, acc);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const Moments mo = moments_of(acc[j]);
                        const Stats st = stats_from(mo, sh);
                        const bool vy_ok = st.vy >= 0.f;                     // clamp(min=0) passes the gradient at 0
                        const float2 vk = max2(st.vk, 0.f);
                        const float vy = fmaxf(st.vy, 0.f);
                        const float2 A1 = fma2(st.mu, bcast(2.f * st.muy), bcast(p.C1));
                        const float2 B1 = fma2(st.mu, st.mu, bcast(fmaf(st.muy, st.muy, p.C1)));
                        const float2 A2 = fma2(bcast(2.f), st.cov, bcast(p.C2));
                        const float2 B2 = add2(vk, bcast(vy + p.C2));
                        const float2 R1 = rcp2(B1), R2 = rcp2(B2);
                        const float2 Cs = mul2(A2, R2);
                        const float2 L = mul2(A1, R1);
                        const float2 S = mul2(L, Cs);
                        const float2 ch = mul2(L, R2);
                        const float2 sr2 = mul2(S, R2);
                        const float2 nbv = f2(vy_ok ? sr2.x : 0.f, vy_ok ? sr2.y : 0.f);
                        float2 a = mul2(mul2(Cs, R1), fma2(L, bcast(-st.muy), st.mu));
                        a = fma2(nbv, bcast(mo.my + sh.ecy), a);
                        a = fma2(ch, fma2(mo.mk, bcast(-1.f), sh.nec), a);
                        ab[j] = f2(a.x + a.y, nbv.x + nbv.y);
                        cc[j] = ch;
                        if (ZMODE) {
                            // predicated adds (never a multiply by 0: the window columns past the strip are computed on
                            // never-written pad columns of vbuf whose stale bits can be NaN / Inf)
                            if ((zmh >> j) & 1u) {
                                z_ss = add2(z_ss, S);
                                if (ZMODE == 1) {               // ZMODE 2: the training objective reads the SSIM means only
                                    z_cs = add2(z_cs, Cs);
                                    z_sg = add2(z_sg, max2(vk, 1e-4f));
                                }
                            }
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) ab[j] = cc[j] = f2(0.f, 0.f);
                }
                float4* d0 = reinterpret_cast<float4*>(sm.cbuf[b & 1] + ho * kCPitch + hg * 8 + half * 4);
                float4* d1 = reinterpret_cast<float4*>(sm.cbuf[b & 1] + ho * kCPitch + kTWI + hg * 8 + half * 4);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    d0[j] = make_float4(ab[2 * j].x, ab[2 * j].y, ab[2 * j + 1].x, ab[2 * j + 1].y);
                    d1[j] = make_float4(cc[2 * j].x, cc[2 * j].y, cc[2 * j + 1].x, cc[2 * j + 1].y);
                }
            }
            if (b + 2 < nb) nb_arrive(NB_VEMPTY + (b & 1));
            nb_arrive(NB_CFULL + (b & 1));
        }
        zv[0] = (double)z_ss.x; zv[1] = (double)z_ss.y; zv[2] = (double)z_cs.x; zv[3] = (double)z_cs.y;
        zv[4] = (double)z_sg.x; zv[5] = (double)z_sg.y;
    } else if (grp == 2) {
        // =========================================================== G2: Sobel / pixel adjoint S(b) -> gbuf[b & 1]
        const float npx = (float)p.B * (float)p.H * (float)p.W;
        const float k_pix = g_pix * p.w_pixel / npx * (p.pixel_combine == MMIF_COMBINE_MAX ? 1.f : 0.5f);
        const float k_grad = g_grad * p.w_grad / npx * (p.grad_combine == MMIF_COMBINE_MAX ? 1.f : 0.5f);
        // Sobel-adjoint phase: column of this thread and its sliding state (see fusion_loss_bwd_kernel)
        const int s_ci = 30 * warp + lane - 1;
        const int s_c = j0 + s_ci;
        const bool s_colok = (s_c >= 0) && (s_c < p.W) && (s_ci <= kTG);
        const bool s_own = (lane >= 1) && (lane <= 30) && (s_ci >= 0) && (s_ci < kTG) && (s_c < jend);
        const int s_cc = min(max(s_c, 0), p.W - 1);
        const int s_t0 = min(s_cc - jw0, kRPB - 1);
        const int s_tm = min(((s_cc == 0) ? 1 : s_cc - 1) - jw0, kRPB - 1);
        const int s_tp = min(((s_cc == p.W - 1) ? p.W - 2 : s_cc + 1) - jw0, kRPB - 1);
        constexpr int kRingImg = kWsRows * kRPB;
        const bool s_strip_int = (j0 >= 3) && (j0 + kTG <= p.W - 3);
        const float* s_p0 = &sm.ring[0][0][min(max(s_c - jw0, 1), kRPB - 2)];
        const float s_ownf = s_own ? 1.f : 0.f;
        const int s_gcol = s_own ? s_ci : 0;
        float2 s_dA = f2(0.f, 0.f), s_dB = s_dA, s_sA = s_dA, s_sB = s_dA, s_ucA = s_dA, s_ucB = s_dA;
        float s_dAy = 0.f, s_dBy = 0.f, s_sAy = 0.f, s_sBy = 0.f, s_ucAy = 0.f, s_ucBy = 0.f;
        float s_hxA = 0.f, s_hxB = 0.f, s_vyA = 0.f, s_vyB = 0.f;
        float z_pix = 0.f, z_grad = 0.f;

        int slot = 0;                                   // b % kWsSlots
        mbar_wait_wd(&sm.ring_full[0], 0);
        mbar_wait_wd(&sm.ring_full[1], 0);
        for (int b = 0; b < nb; ++b) {
            const int Rb = R0 + b * kRB;
            mbar_wait_wd(&sm.ring_full[(slot + 2) % kWsSlots], ((b + 2) / kWsSlots) & 1);
            const int rbase = slot * kRB;               // ring row of input row Rb
            if (b >= 2) nb_sync(NB_GEMPTY + (b & 1));             // B2(b - 2) has read this gbuf slot
            float (*gb)[kTMC + 4] = sm.gbuf[b & 1];
            const bool s_fast = !MMIF_WS_NO_SFAST && FAST && s_strip_int && (Rb >= max(2, i0)) && (Rb + 9 <= min(iend, p.H - 1));
            if (s_fast) {
                // two passes of four rows through one copy of the code (instruction footprint, see G1); within a pass the
                // three stages (loads + Sobel + sign factors, neighbour exchange, vertical combination) keep four
                // independent row chains in flight
                // input rows Rb + 2 .. Rb + 9: six in this batch's ring slot, two in the next one; per pass two base pointers
                // with constant row offsets instead of a wrap per row
                const float* ps0 = s_p0 + rbase * kRPB;
                const float* ps1 = s_p0 + ((slot + 1 == kWsSlots) ? 0 : slot + 1) * (kRB * kRPB);
#pragma unroll 1
                for (int h4 = 0; h4 < 2; ++h4) {
                    float tx[4], ty[4], pg[4];
                    const float* plo = ps0 + (2 + 4 * h4) * kRPB;
                    const float* phi = h4 ? ps1 - 2 * kRPB : plo;
#pragma unroll
                    for (int s4 = 0; s4 < 4; ++s4) {
                        const float* rp = (s4 < 2 ? plo : phi) + s4 * kRPB;        // ring row of input row Rb + 2 + 4 h4 + s4
                        const float2 um = f2(rp[-1], rp[kRingImg - 1]);
                        const float2 uc = f2(rp[0], rp[kRingImg]);
                        const float2 up = f2(rp[1], rp[kRingImg + 1]);
                        const float umy = rp[2 * kRingImg - 1], ucy = rp[2 * kRingImg], upy = rp[2 * kRingImg + 1];
                        const float2 d = fma2(bcast(-1.f), um, up);
                        const float2 sv = fma2(bcast(2.f), uc, add2(um, up));
                        const float2 gx = fma2(bcast(2.f), s_dB, add2(s_dA, d));
                        const float2 gy = fma2(bcast(-1.f), s_sA, sv);
                        const float dy = upy - umy;
                        const float sy = fmaf(2.f, ucy, umy + upy);
                        const float gxy = fmaf(2.f, s_dBy, s_dAy + dy);
                        const float gyy = sy - s_sAy;
                        const float S1 = fabsf(gx.x) + fabsf(gy.x), S2 = fabsf(gx.y) + fabsf(gy.y), Sy = fabsf(gxy) + fabsf(gyy);
                        const float D = Sy - fmaxf(S1, S2);
                        const float r = mulsign(k_grad, D);
                        tx[s4] = mulsign(r, gxy);
                        ty[s4] = mulsign(r, gyy);
                        const float dp = s_ucAy - fmaxf(s_ucA.x, s_ucA.y);
                        pg[s4] = mulsign(k_pix, dp);
                        if (ZMODE) {
                            z_grad = fmaf(s_ownf, fabsf(D), z_grad);
                            z_pix = fmaf(s_ownf, fabsf(dp), z_pix);
                        }
                        s_dA = s_dB; s_dB = d; s_sA = s_sB; s_sB = sv; s_dAy = s_dBy; s_dBy = dy; s_sAy = s_sBy; s_sBy = sy;
                        s_ucA = s_ucB; s_ucB = uc; s_ucAy = s_ucBy; s_ucBy = ucy;
                    }
#pragma unroll
                    for (int s4 = 0; s4 < 4; ++s4) {
                        const float txl = __shfl_up_sync(0xffffffffu, tx[s4], 1), txr = __shfl_down_sync(0xffffffffu, tx[s4], 1);
                        const float tyl = __shfl_up_sync(0xffffffffu, ty[s4], 1), tyr = __shfl_down_sync(0xffffffffu, ty[s4], 1);
                        tx[s4] = txl - txr;
                        ty[s4] = fmaf(2.f, ty[s4], tyl + tyr);
                    }
#pragma unroll
                    for (int s4 = 0; s4 < 4; ++s4) {
                        const float hx = tx[s4], vy = ty[s4];
                        if (s_own) gb[h4 * 4 + s4][s_gcol] = (s_hxA + s_vyA) + fmaf(2.f, s_hxB, hx - vy) + pg[s4];
                        s_hxA = s_hxB; s_hxB = hx; s_vyA = s_vyB; s_vyB = vy;
                    }
                }
            } else {
#pragma unroll 4
                for (int step = 0; step < kRB; ++step) {
                    const int qp = Rb + 2 + step;
                    int rr = (qp < 0) ? -qp : ((qp >= p.H) ? 2 * p.H - 2 - qp : qp);
                    const int lr = (min(max(rr - R0, b * kRB), b * kRB + 3 * kRB - 1)) % kWsRows;
                    const float2 um = f2(sm.ring[0][lr][s_tm], sm.ring[1][lr][s_tm]);
                    const float2 uc = f2(sm.ring[0][lr][s_t0], sm.ring[1][lr][s_t0]);
                    const float2 up = f2(sm.ring[0][lr][s_tp], sm.ring[1][lr][s_tp]);
                    const float umy = sm.ring[2][lr][s_tm], ucy = sm.ring[2][lr][s_t0], upy = sm.ring[2][lr][s_tp];
                    const float2 d = fma2(bcast(-1.f), um, up);
                    const float2 sv = fma2(bcast(2.f), uc, add2(um, up));
                    const float2 gx = fma2(bcast(2.f), s_dB, add2(s_dA, d));
                    const float2 gy = fma2(bcast(-1.f), s_sA, sv);
                    const float dy = upy - umy;
                    const float sy = fmaf(2.f, ucy, umy + upy);
                    const float gxy = fmaf(2.f, s_dBy, s_dAy + dy);
                    const float gyy = sy - s_sAy;
                    const int qt = qp - 1;
                    float tx = 0.f, ty = 0.f;
                    if (s_colok && qt >= 0 && qt < p.H) {
                        const float S1 = fabsf(gx.x) + fabsf(gy.x), S2 = fabsf(gx.y) + fabsf(gy.y), Sy = fabsf(gxy) + fabsf(gyy);
                        float r;
                        if (FAST) r = mulsign(k_grad, Sy - fmaxf(S1, S2));
                        else if (p.grad_combine == MMIF_COMBINE_MAX) r = k_grad * norm_der(Sy - fmaxf(S1, S2), p.grad_norm);
                        else r = k_grad * (norm_der(Sy - S1, p.grad_norm) + norm_der(Sy - S2, p.grad_norm));
                        tx = mulsign(r, gxy);
                        ty = mulsign(r, gyy);
                        if (ZMODE && s_own && qt >= i0 && qt < iend) {
                            if (FAST || p.grad_combine == MMIF_COMBINE_MAX) z_grad += norm_val(Sy - fmaxf(S1, S2), FAST ? MMIF_NORM_L1 : p.grad_norm);
                            else z_grad += 0.5f * (norm_val(Sy - S1, p.grad_norm) + norm_val(Sy - S2, p.grad_norm));
                        }
                    }
                    const float txl = __shfl_up_sync(0xffffffffu, tx, 1), txr = __shfl_down_sync(0xffffffffu, tx, 1);
                    const float tyl = __shfl_up_sync(0xffffffffu, ty, 1), tyr = __shfl_down_sync(0xffffffffu, ty, 1);
                    float hx = txl - txr, vy = tyl + 2.f * ty + tyr;
                    if (s_c == 1) { hx -= txl; vy += tyl; }
                    if (s_c == p.W - 2) { hx += txr; vy += tyr; }
                    const int gi = qp - 2;
                    float G = s_hxA + 2.f * s_hxB + hx + s_vyA - vy;
                    if (gi == 1) G += s_hxA - s_vyA;
                    if (gi == p.H - 2) G += hx + vy;
                    if (FAST) G += mulsign(k_pix, s_ucAy - fmaxf(s_ucA.x, s_ucA.y));
                    else if (p.pixel_combine == MMIF_COMBINE_MAX) G += k_pix * norm_der(s_ucAy - fmaxf(s_ucA.x, s_ucA.y), p.pixel_norm);
                    else G += k_pix * (norm_der(s_ucAy - s_ucA.x, p.pixel_norm) + norm_der(s_ucAy - s_ucA.y, p.pixel_norm));
                    if (s_own && gi >= i0 && gi < iend) {
                        gb[step][s_ci] = G;
                        if (ZMODE) {
                            if (FAST || p.pixel_combine == MMIF_COMBINE_MAX) z_pix += norm_val(s_ucAy - fmaxf(s_ucA.x, s_ucA.y), FAST ? MMIF_NORM_L1 : p.pixel_norm);
                            else z_pix += 0.5f * (norm_val(s_ucAy - s_ucA.x, p.pixel_norm) + norm_val(s_ucAy - s_ucA.y, p.pixel_norm));
                        }
                    }
                    s_dA = s_dB; s_dB = d; s_sA = s_sB; s_sB = sv; s_dAy = s_dBy; s_dBy = dy; s_sAy = s_sBy; s_sBy = sy;
                    s_hxA = s_hxB; s_hxB = hx; s_vyA = s_vyB; s_vyB = vy;
                    s_ucA = s_ucB; s_ucB = uc; s_ucAy = s_ucBy; s_ucBy = ucy;
                }
            }
            nb_arrive(NB_GFULL + (b & 1));
            mbar_arrive(&sm.ring_empty[slot]);            // S never looks at input rows before Rb again
            slot = (slot + 1 == kWsSlots) ? 0 : slot + 1;
        }
        zv[6] = (double)z_pix; zv[7] = (double)z_grad;
    } else {
        // =========================================================== G3: vertical adjoint B1(b) (stateful) -> tbuf, horizontal adjoint + combine + store B2(b)
        const int ho = lane & 7, hg = warp * 4 + (lane >> 3);
        const float k_ssim2 = 2.f * g_ssim * p.ssim_base / ((float)p.Hout * (float)p.Wout);
        const bool b1_valid = (jw0 + kVOFF + t >= 0) && (jw0 + kVOFF + t < p.Wout);      // window column t exists in the image
        float2 carry[HALO][2];
#pragma unroll
        for (int d = 0; d < HALO; ++d) carry[d][0] = carry[d][1] = f2(0.f, 0.f);
        int slot = 0;
        for (int b = 0; b < nb; ++b) {
            const int Rb = R0 + b * kRB;
            const bool emit = (Rb + kRB > i0);
            nb_sync(NB_CFULL + (b & 1));
            {
                const float2* cb = sm.cbuf[b & 1];
                float2 P[kRB + HALO][2];
#pragma unroll
                for (int d = 0; d < kRB + HALO; ++d) {
                    P[d][0] = (d < HALO) ? carry[d][0] : f2(0.f, 0.f);
                    P[d][1] = (d < HALO) ? carry[d][1] : f2(0.f, 0.f);
                }
#pragma unroll
                for (int r = 0; r < kRB; ++r) {
                    const float2 v0 = cb[r * kCPitch + t];
                    const float2 v1 = cb[r * kCPitch + kTWI + t];
#pragma unroll
                    for (int d = 0; d < WIN; ++d) {
                        P[r + d][0] = fmas(p.taps.w[d], v0, P[r + d][0]);
                        P[r + d][1] = fmas(p.taps.w[d], v1, P[r + d][1]);
                    }
                }
                if (b + 2 < nb) nb_arrive(NB_CEMPTY + (b & 1));
                if (emit) {
                    if (b1_valid) {
#pragma unroll
                        for (int o = 0; o < kRB; ++o) {
                            sm.tbuf[o * kCPitch + t] = P[o][0];
                            sm.tbuf[o * kCPitch + kTWI + t] = P[o][1];
                        }
                    } else {                      // a window column outside the image contributes nothing
#pragma unroll
                        for (int o = 0; o < kRB; ++o) {
                            sm.tbuf[o * kCPitch + t] = f2(0.f, 0.f);
                            sm.tbuf[o * kCPitch + kTWI + t] = f2(0.f, 0.f);
                        }
                    }
                }
#pragma unroll
                for (int d = 0; d < HALO; ++d) { carry[d][0] = P[d + kRB][0]; carry[d][1] = P[d + kRB][1]; }
            }
            group_sync(NB_TBUF);                          // tbuf written
            nb_sync(NB_GFULL + (b & 1));                  // S(b) has written gbuf[b & 1]
            if (emit) {
                const int i = Rb + ho;
                if (i >= i0 && i < iend && hg * 8 < kTG && j0 + hg * 8 < jend) {
                    mbar_wait_wd(&sm.ring_full[slot], (b / kWsSlots) & 1);
                    float2 acc[8][2];
                    hpass<WIN, 2, true>(sm.tbuf + ho * kCPitch + hg * 8, kTWI, p.taps, acc);
                    const int lr = slot * kRB + ho;
                    float outv[8], u1[8], u2[8], uy[8], gbv[8];
                    {
                        const int tc = kOFF + hg * 8;
                        const float4* q1 = reinterpret_cast<const float4*>(&sm.ring[0][lr][tc]);
                        const float4* q2 = reinterpret_cast<const float4*>(&sm.ring[1][lr][tc]);
                        const float4* qy = reinterpret_cast<const float4*>(&sm.ring[2][lr][tc]);
                        const float4* qg = reinterpret_cast<const float4*>(&sm.gbuf[b & 1][ho][hg * 8]);
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const float4 a = q1[h], bq = q2[h], c = qy[h], g4 = qg[h];
                            u1[4 * h] = a.x; u1[4 * h + 1] = a.y; u1[4 * h + 2] = a.z; u1[4 * h + 3] = a.w;
                            u2[4 * h] = bq.x; u2[4 * h + 1] = bq.y; u2[4 * h + 2] = bq.z; u2[4 * h + 3] = bq.w;
                            uy[4 * h] = c.x; uy[4 * h + 1] = c.y; uy[4 * h + 2] = c.z; uy[4 * h + 3] = c.w;
                            gbv[4 * h] = g4.x; gbv[4 * h + 1] = g4.y; gbv[4 * h + 2] = g4.z; gbv[4 * h + 3] = g4.w;
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float x1s = u1[j] - sh.c.x;
                        const float x2s = u2[j] - sh.c.y;
                        const float ys = uy[j] - sh.cy;
                        const float dS = fmaf(x2s, acc[j][1].y, fmaf(x1s, acc[j][1].x, fmaf(-ys, acc[j][0].y, acc[j][0].x)));
                        outv[j] = fmaf(k_ssim2, dS, gbv[j]);
                    }
                    float* dst = p.dF + img_off + (size_t)i * p.W + j0 + hg * 8;
                    if (p.vec_store && j0 + hg * 8 + 8 <= jend) {
                        reinterpret_cast<float4*>(dst)[0] = make_float4(outv[0], outv[1], outv[2], outv[3]);
                        reinterpret_cast<float4*>(dst)[1] = make_float4(outv[4], outv[5], outv[6], outv[7]);
                    } else if (p.vec_store && j0 + hg * 8 + 4 == jend) {
                        reinterpret_cast<float4*>(dst)[0] = make_float4(outv[0], outv[1], outv[2], outv[3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (j0 + hg * 8 + j < jend) dst[j] = outv[j];
                    }
                }
            }
            if (b + 2 < nb) nb_arrive(NB_GEMPTY + (b & 1));
            mbar_arrive(&sm.ring_empty[slot]);            // input rows of batch b are free
            group_sync(NB_TBUF);                          // tbuf may be rewritten
            slot = (slot + 1 == kWsSlots) ? 0 : slot + 1;
        }
    }
    if (ZMODE) cta_finish<kWsNT>(p.fin, zv, sm.red, &sm.flag, n, blk, nblk);
}

}  // namespace mmif
