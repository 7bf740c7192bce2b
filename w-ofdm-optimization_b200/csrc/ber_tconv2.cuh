// ber_tconv2.cuh -- K1, second generation of the tensor-core-convolution frame kernel (tcgen05, sm_100a).
//
// Same chain as ber_frame_kernel (ber_kernel.cuh; reference loop body python/ofdm_utils/wofdm_simulation.py:171-240,
// matlab/main_BER_calculation.m:245-273) and the same Hankel-operand convolution as ber_tconv.cuh (the frame stream,
// split in two fp16 halves, IS the K-major A operand; the frame's taps are B; fp32 accumulators in tensor memory).
// What is new is everything around the convolution -- the first generation spent 65 % of its issue slots there:
//
//   * ONE pass over the accumulators, and the noise where the receiver needs it.  Every receiver thread draws, into
//     registers and while the MMAs run, the noise of exactly the samples its FFT rows will gather (plus its share of the
//     symbol's other samples, which only count in the noise power; ber_kernel.cuh: noise_draw48 is the numbering).  When
//     the MMAs have completed, tcgen05.ld reads r = conv(h, u) once: |r|^2 goes into the frame-wide sum and r itself, as
//     plain fp32, over the dead split stream (two interleaved halves: conflict-free stores, base + immediate loads).  The
//     exact-SNR gain g = sqrt(Pr 10^(-snr/10) / Pn) (wofdm_simulation.py:135-138) is applied where the receiver gathers
//     its block: y = r + g n.  The first generation's second tcgen05.ld pass, its y store and one CTA barrier per frame
//     are gone.
//   * Symbols are level codes (ber_kernel.cuh: load_sym_idx): the slicer's packed decisions are compared with the sent
//     codes directly, no decision table, bit errors by the GF(2)-linear Gray map of the XOR.
//   * 48 random bits per complex noise sample instead of 64: a 32-bit radius word and a 16-bit angle (65 536 phases),
//     three Philox4x32-10 calls per eight samples.
//   * A dedicated ninth (seventeenth) warp issues the MMAs: it alone waits for the whole stream to be written (bar.sync)
//     and then sits in front of the tensor core's queue, while the working warps announce their part (bar.arrive) and
//     draw their noise.  MMA descriptors advance by one addition.
//
// fp32; N = 256: one CTA of 256 threads per frame, two CTAs per SM (256 of the 512 tensor-memory columns each);
// N = 512: one CTA of 512 threads per frame and SM.  S <= 16 symbols in one Tx pass, L <= LB (21 or 84), prefix / suffix /
// tails within the outer register rows (ber_host.cu:choose_variant checks).
#pragma once
#include <cuda_fp16.h>
#include <cstdio>
#include "ber_kernel.cuh"
#include "ber_tconv.cuh"

namespace wofdm {

// transform group `slot` of a CTA works on its OFDM symbol S - 1 - slot: the pilot (symbol 0), whose receiver everybody waits
// for, then sits in the warp with the highest index, which the warp schedulers serve first
#ifndef TCV2_REVERSE_SLOTS
#define TCV2_REVERSE_SLOTS 1
#endif
#define TCV2_SLOT_SYMBOL(slot, S) (TCV2_REVERSE_SLOTS ? (S) - 1 - (slot) : (slot))
// development aid: per-warp clock() stamps at the phase boundaries of a few frames of CTA 0, printed from the device
#ifndef TCV2_TRACE
#define TCV2_TRACE 0
#endif
#if TCV2_TRACE
#define TCV2_STAMP(k) do { if (trace_on && lane == 0) trace_buf[warp * 12 + (k)] = clock64(); } while (0)
#else
#define TCV2_STAMP(k) do { } while (0)
#endif
#ifndef TCV2_GT
#define TCV2_GT 3
#endif
// Slicer folded into the equaliser product (production instantiations): the taps are stored halved, so the scale and offset
// of slice_index (y = e / 2 + (m - 2) / 2) ride on the complex product's first packed FMA, and the upper clamp is taken in
// floating point (FMNMX, one issue cycle) before the saturating round-up conversion instead of on the integers afterwards.
// Same decisions as slice_index up to the rounding of the fused sum (fp32 grade either way; ties still go to the lower level).
// Measured: 16 packed instructions and 32 two-cycle integer clamps fewer per thread and frame, 5.76 ms against 5.78 per
// 202 500 frames -- within the noise, so the build keeps slice_index (one definition of the decision for every kernel).
#ifndef TCV2_FOLD_SLICER
#define TCV2_FOLD_SLICER 0
#endif
#ifndef TCV2_TXY_U
#define TCV2_TXY_U 8      // stream samples per thread and round of the masked chain's loader (tconv2_load_masked)
#endif
#ifndef TCV2_DEBUG_BARRIERS
#define TCV2_DEBUG_BARRIERS 0          // 1 (libwofdm_dbg.so): every relaxed synchronisation of the kernel replaced by a full barrier --
#endif                                 // the reference the race test compares the production build with (compute-sanitizer is closed here)
// Kernels whose working warps issue the MMAs (N = 1024): 1 = the issue is staggered over all warps -- four groups of four
// warps issue a quarter of the tiles each, group g after g quarters of its noise draws -- so nobody sits in front of the
// tensor core's queue for the whole convolution.  Each group has its own "stream complete" named barrier (14 - g).
#ifndef TCV2_STAGGER
#define TCV2_STAGGER 0     // (measured: 10.97 ms against 10.84 with the issuers skipping the accumulator pass -- the kernel is throughput bound)
#endif
#ifndef TCV2_REBALANCE
#define TCV2_REBALANCE 1
#endif
// The frame's tiles complete in tconv2_nseg(N) segments, one mbarrier each: the accumulator pass starts on the first tiles while
// the tensor core still works on the last ones.  Segment k is signalled once tile seg_end(k) -- the first tile of the NEXT
// segment -- is complete too: that tile reads the last PAD samples of its predecessor's stream as convolution history, and
// r is parked over the stream.
// Measured (ms per launch, one against three segments): N = 512: 4.55 -> 4.41 (the MMAs outlast the noise draws there);
// N = 256: 5.79 -> 5.88 (they do not: only the extra waits remain); N = 1024: 10.83 either way.
#ifndef TCV2_NSEG_512
#define TCV2_NSEG_512 3
#endif
constexpr int TCV2_MAXSEG = 4;
__host__ __device__ constexpr int tconv2_nseg(int N) { return N == 512 ? TCV2_NSEG_512 : 1; }
__host__ __device__ constexpr int tconv2_seg_end(int nseg, int ntile, int k) { return (ntile * (k + 1) + nseg - 1) / nseg; }   // tiles < seg_end(k): segments 0..k
__host__ __device__ constexpr int tconv2_seg_of(int nseg, int ntile, int tt) {
    int k = 0;
    while (k < nseg - 1 && tt >= tconv2_seg_end(nseg, ntile, k)) ++k;
    return k;
}
constexpr int TCV2_BAR_STREAM = 14;      // named barrier: "the split stream of this frame is complete"
constexpr int TCV2_BAR_RES = 15;         // named barrier of the working warps before a flush of the resolved counters (RES)

// N <= 512: the CTA has one more warp that only issues the MMAs.  The register file then leaves the working threads 96
// registers (two CTAs of 288 threads, or one of 544, per SM), which the N = 256 kernel fits without spills and the N = 512
// kernel with ~60 bytes of them (measured: 2.06e8 -> 2.12e8 OFDM symbols/s all the same).  N = 1024 (clusters) spills
// 200 bytes under that cap (8.6e7 -> 6.8e7), so there four of the working warps, rotating from frame to frame, issue a
// quarter of the frame's MMAs each before they draw their noise.
#ifndef TCV2_MMAW_MAXN
#define TCV2_MMAW_MAXN 512
#endif
// Register reallocation (setmaxnreg): the MMA warp is launched inside a whole warp group of four (setmaxnreg is a warp-group
// instruction: with an incomplete group -- the MMA warp and one idle warp were tried -- the release never completes and the
// working warps spin in their request); the three other warps are idle register donors.  The group shrinks to 24 registers
// and the working warps grow from what the launch grants to tconv2_work_regs: NT = 256: 384 threads x 80 at launch ->
// 256 x 104 + 128 x 24 (5.91 -> 5.83 ms per 202 500 frames).  The donors walk through the MMA warp's barrier
// sequence and issue nothing.
#ifndef TCV2_SETMAXNREG
#define TCV2_SETMAXNREG 1
#endif
// (NT = 512: measured slower, 4.64 ms against 4.51 per 60 000 frames -- 20 warps of 112 registers against 17 of 96 with ~60
//  bytes of spills; it keeps the lone MMA warp)
#ifndef TCV2_SETMAXNREG_1024
#define TCV2_SETMAXNREG_1024 0     // (measured: 104 bytes of spills at 112 registers, 11.85 ms against 11.22)
#endif
__host__ __device__ constexpr bool tconv2_setmaxnreg(int N, int NT) { return TCV2_SETMAXNREG && (NT == 256 || (TCV2_SETMAXNREG_1024 && N == 1024)); }
__host__ __device__ constexpr int tconv2_mma_warp_threads(int N, int NT) {
    return tconv2_setmaxnreg(N, NT) ? 128 : (N <= TCV2_MMAW_MAXN && NT <= 512) ? 32 : 0;
}
__host__ __device__ constexpr int tconv2_work_regs(int NT) { return NT == 256 ? 104 : 112; }   // (NT = 512: 640 x 96 -> 512 x 112 + 128 x 24)
// (Registers: ptxas derives 96 per thread from __launch_bounds__(288, 2) and that is what the hardware grants -- the register
//  file is allocated to an even number of warps per CTA: a build forced to 112 registers ran one CTA per SM, 7.9 ms instead
//  of 6.0, and the 544-thread kernel at 117 failed to launch.)
constexpr int TCV2_NISSUE = 4;
// Taps: the Hankel operand's row r holds the samples 4r - PAD .. 4r + 3, PAD = LB - 1 rounded up to 4 (r stays 16-byte
// aligned behind the pad): (PAD + 4) / 8 K steps of 16 halves, two MMAs (hi, lo stream half) each.  LB = 21: PAD 20, 3 K
// steps, 6 MMAs per tile of 512 samples; LB = 84 (configs[4] "optionally 84 taps"): PAD 84, 11 K steps, 22 MMAs.
__host__ __device__ constexpr int tconv2_pad(int LB) { return (LB - 1 + 3) & ~3; }
__host__ __device__ constexpr int tconv2_ksteps(int LB) { return (tconv2_pad(LB) + 4) / 8; }
__host__ __device__ constexpr int tconv2_tbl(int LB) { return (tconv2_pad(LB) + 4) / 4 * 128; }   // bytes of one taps table (8 columns x K halves)
__host__ __device__ constexpr int tconv2_zero(int LB) { return (LB - 1 + 3 + 4) & ~3; }             // zero samples written behind the stream
// |n|^2 of a thread's extras of level 2 and above (words V[3j .. 3j+2] of pair j >= 1, ber_kernel.cuh: noise_draw48): they
// only count in the noise power.  Kept out of line: the common shapes have at most two levels and the kernel is register bound.
__device__ __forceinline__ float2 n48_more_extras(const BerParams& prm, long long f, uint32_t q0, int var, int nlev, int xt, int tpf, int xas) {
    float2 pnx = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int jp = 1; 2 * jp < nlev; ++jp) {
        const int w0 = 3 * jp;
        const uint4 ca = noise48_call(prm, f, q0 + 6 + (uint32_t)(w0 >> 2), var);
        const uint4 cb = noise48_call(prm, f, q0 + 6 + (uint32_t)((w0 + 2) >> 2), var);
        const uint32_t aw = u4_word(ca, w0 & 3), u0 = u4_word((w0 + 1) >> 2 == w0 >> 2 ? ca : cb, (w0 + 1) & 3), u1 = u4_word(cb, (w0 + 2) & 3);
        float2 e2, e3;
        gauss_quad48(u0, u1, aw, e2, e3);
        if (xt + 2 * jp * tpf < xas) pnx = csq_acc(e2, pnx);
        if (xt + (2 * jp + 1) * tpf < xas) pnx = csq_acc(e3, pnx);
    }
    return pnx;
}
__host__ __device__ constexpr int tconv2_wtx_len(int stride, int tail_tx) { return (stride + tail_tx + 3) & ~3; }
__host__ __device__ constexpr int tconv2_wrx_len(int N, int tail_rx) { return (N + tail_rx + 3) & ~3; }

// Channel-mask chain (TXY instantiations): the frame's serialised Tx stream gathered from the mask product's output
// (mask_gemm.cu, BerParams::tx_y: column s of the frame = the filtered symbol f_s, n_tx samples (Re, Im) interleaved, the
// filter tail of symbol s-1 already inside, main_channel_mask.m:413-416).  The filtered symbols are overlap-added with the
// frame stride (tx2rx, :420-431): stream[s stride + i] = f_s[i] + f_{s-1}[stride + i].  TCV2_TXY_U stream samples per thread
// and round, two loads each in flight (the loader is latency bound otherwise).
template <int NT>
static __device__ __forceinline__ void tconv2_load_masked(const float* __restrict__ y0, int yp, int S, int stride, int n_tx, int body,
                                                          uint32_t* __restrict__ uh, uint32_t* __restrict__ ul, int tid) {
    constexpr int U = TCV2_TXY_U;
    for (int p0 = tid; p0 < body; p0 += U * NT) {
        float2 a[U], c[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = p0 + u * NT;
            a[u] = c[u] = make_float2(0.f, 0.f);
            if (p < body) {
                const int s = min(p / stride, S), i = p - s * stride;
                const float* ys = y0 + (size_t)s * yp;
                if (s < S) a[u] = __ldg(reinterpret_cast<const float2*>(ys + 2 * i));
                if (s >= 1 && stride + i < n_tx) c[u] = __ldg(reinterpret_cast<const float2*>(ys - yp + 2 * (stride + i)));
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = p0 + u * NT;
            if (p < body) {
                uint32_t hi, lo;
                split_h2(cscale(TCV_XSCALE, cadd(a[u], c[u])), hi, lo);
                uh[p] = hi; ul[p] = lo;
            }
        }
    }
}

template <int N, int NT, int NTILE, int LB = TCV_LB, bool RES = false>
__host__ __device__ inline BerSmem tconv2_smem_layout(int S, int stride, int tail_tx, int tail_rx, int L, int nvar, int use_global) {
    using P = FftPlan<N>;
    constexpr int FPP = NT / P::TPF;
    BerSmem m;
    m.pad = tconv2_pad(LB);
    m.flen = tconv2_pad(LB) + NTILE * 512;
    m.xlen = FPP * P::XLEN;
    int o = 0;
    o += m.flen * 4;                 m.off_lo = o;        // ahi
    o += m.flen * 4;                                      // alo (r lies over ahi | alo from byte 4 * TCV_PAD, two halves of
    o += 64;                                              //      128 NTILE + 4 chunks of 16 bytes)
    o = (o + 15) & ~15;              m.off_x = o;
    o += m.xlen * 8;                 m.off_tw = o;
    o += P::NTW * 8;                 m.off_geq = o;
    o += N * 8;                      m.off_bt = o;
    o += 4 * tconv2_tbl(LB);         m.off_wtx = o;       // taps blocks [A0 | A1 | B0 | B1] (below), 8 columns x K halves each
    const int nv = nvar > 1 ? nvar : 1;                   // window pairs evaluated per frame (BerParams::nvar)
    o += nv * tconv2_wtx_len(stride, tail_tx) * 4;   m.off_wrx = o;
    o += nv * tconv2_wrx_len(N, tail_rx) * 4;        m.off_red = o;
    o += 64 * 4;                              m.off_qlut = o;
    o += 2 * 256 * 8;                         m.off_gmask = o;      // lattice points: Rx (pilot) copy, Tx copy (carries the flat window value)
    o += P::TPF * 32;                         m.off_symw = o;
    o += S * P::TPF * 16;                     m.off_bar = o;
    o += 8 * TCV2_MAXSEG + 8;
    m.off_res = 0;
    if constexpr (RES) { o = (o + 15) & ~15; m.off_res = o; o += nv * N * 8; }   // per-sub-carrier error accumulators
    m.off_hf = m.off_taps = m.off_dlut = 0;
    m.bytes = ((size_t)o + 15) & ~(size_t)15;
    (void)L; (void)use_global;
    return m;
}

// CL = 2: a thread-block cluster of two CTAs shares one frame, S/2 consecutive OFDM symbols and their part of the frame
// stream per CTA (N = 1024: stream and exchange buffers of a whole frame are 278 KB, more than one SM holds).  The CTAs meet
// three times per frame through distributed shared memory: the second CTA takes the first one's last Tx tail and the
// L - 1 samples of convolution history (PULLED, a few dozen words), the per-warp power partials and the pilot's equaliser
// taps are PUSHED into both CTAs, so every read is local.
// RES: error counters resolved by sub-carrier and / or channel (BerParams::res_chan / res_bins, ber_kernel.cuh: res_flush);
// in a cluster every CTA keeps and flushes the accumulators of its own symbols
// HS: the frame loop of the common shape class compiled with its switches as constants (ber_host.cu: tconv2_fixed_shape):
// a flat Tx window with cp, cs >= tail_tx, tail_rx = 0, one window pair, no guard band, the symbols drawn in the kernel.
// N, S, L, the Rx window's flatness and the conventions (noise_norm, constellation) stay run-time.
template <int N, int NT, int NTILE, int MINB, bool VERIFY, int CL = 1, int LB = TCV_LB, bool TXY = false, bool RES = false,
          bool HS = false>
__global__ void __launch_bounds__(NT + tconv2_mma_warp_threads(N, NT), MINB)
ber_tconv2_kernel(const BerParams prm) {
    using T = float;
    using C2 = float2;
    using P = FftPlan<N>;
    constexpr int TPF = P::TPF, FPP = NT / TPF, ER = 2, NW = NT / 32;
    static_assert(NT == 256 || NT == 512, "eight warps read a tile's accumulators");
    constexpr int TG = NT / 256, NTH = (NTILE + TG - 1) / TG;             // tile sets; tiles per thread
    constexpr uint32_t TMEM_COLS = tconv_tmem_cols(NTILE);
    constexpr int NSEG = tconv2_nseg(N);
    static_assert(NSEG <= TCV2_MAXSEG, "one mbarrier per segment");
    static_assert(16 * NTILE <= (int)TMEM_COLS, "accumulators of a frame must fit tensor memory");
    static_assert(CL * NW <= 32, "per-warp power partials of all CTAs must fit the reduction scratch");
    static_assert(!RES || !VERIFY, "resolved counters: production kernels");
    static_assert(!HS || (CL == 1 && !VERIFY && !TXY && !RES), "the fixed-shape frame loop: one-CTA production kernels");

    extern __shared__ __align__(128) unsigned char tcv_smem[];
    unsigned char* const smem_raw = tcv_smem;
    const int tid = threadIdx.x;    // (tried: an identity shuffle to stop ptxas re-deriving the index from %tid.x -- 12 S2R instead of 22, 6.27 ms against 5.79)
    const int warp = tid >> 5, lane = tid & 31;
    const int slot = tid / TPF, t = tid % TPF;
    int rank = 0;
    if constexpr (CL > 1) rank = (int)cooperative_groups::this_cluster().block_rank();
    const bool last_rank = rank == CL - 1;
    const int S = prm.S / CL, sb = rank * S;    // this CTA's symbols: sb .. sb + S - 1 (the whole frame when CL == 1)
    const int stride = prm.stride, n_tx = prm.n_tx, beta = prm.tail_tx, L = prm.L;
    const int cp = prm.cp, cs = prm.cs;
    const int hh = HS ? 0 : prm.tail_rx >> 1;
    const int hb = prm.bits >> 1, m = 1 << hb;
    const int sec = S * stride;                 // samples kept after the channel (this CTA's)
    const int body = beta + sec;                // serialised Tx stream length
    const int npow = (prm.noise_norm == 1 && last_rank) ? body + L - 1 : sec;   // samples inside the frame-wide power sums

    const int nvar = (!VERIFY && !HS && prm.nvar > 1) ? prm.nvar : 1;     // window pairs evaluated on every frame's symbols
    constexpr int PAD = tconv2_pad(LB), KS = tconv2_ksteps(LB), TBL = tconv2_tbl(LB), ZERO = tconv2_zero(LB);
    const BerSmem lay = tconv2_smem_layout<N, NT, NTILE, LB, RES>(S, stride, beta, prm.tail_rx, L, nvar, 0);
    uint32_t* const ahi = reinterpret_cast<uint32_t*>(smem_raw);
    uint32_t* const alo = reinterpret_cast<uint32_t*>(smem_raw + lay.off_lo);
    uint32_t* const uh = ahi + PAD;         // uh[i], ul[i]: split stream sample i
    uint32_t* const ul = alo + PAD;
    C2* const rb = reinterpret_cast<C2*>(smem_raw + PAD * 4);   // channel output r[i], over the dead split stream (keeps ahi's zero pad)
    static_assert((PAD * 4) % 16 == 0, "r is stored in 16-byte pairs");
    C2* const xbuf = reinterpret_cast<C2*>(smem_raw + lay.off_x);  // FFT exchange, one region per transform group
    C2* tw = reinterpret_cast<C2*>(smem_raw + lay.off_tw);
    C2* geq = reinterpret_cast<C2*>(smem_raw + lay.off_geq);
    unsigned char* bt = smem_raw + lay.off_bt;
    T* const wtx_all = reinterpret_cast<T*>(smem_raw + lay.off_wtx);   // [nvar][WTXL]
    T* const wrx_all = reinterpret_cast<T*>(smem_raw + lay.off_wrx);   // [nvar][WRXL]
    const int WTXL = tconv2_wtx_len(stride, beta), WRXL = tconv2_wrx_len(N, prm.tail_rx);
    T* red = reinterpret_cast<T*>(smem_raw + lay.off_red);
    C2* qlut = reinterpret_cast<C2*>(smem_raw + lay.off_qlut);     // level code -> lattice point
    C2* qtx = qlut + 256;                                           // ... times the flat Tx window value
    uint4* gmask = reinterpret_cast<uint4*>(smem_raw + lay.off_gmask);
    uint4* symw = reinterpret_cast<uint4*>(smem_raw + lay.off_symw);
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem_raw + lay.off_bar);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_raw + lay.off_bar + 8 * TCV2_MAXSEG);
    C2* const xb = xbuf + slot * P::XLEN;

    // ---- one-time: tensor memory, barrier, tables ----
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(tcv_smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int k = 0; k < NSEG; ++k)       // one commit per issuing warp, segment and frame
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(tcv_smem_u32(bar + k)), "r"(tconv2_mma_warp_threads(N, NT) ? 1 : (TCV2_STAGGER && !TCV2_DEBUG_BARRIERS) ? NT / 32 : TCV2_NISSUE) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < P::NTW; i += NT) tw[i] = reinterpret_cast<const C2*>(prm.tw)[i];
    // flat windows (host-checked): the Tx window's flat value rides on the constellation table and wtx holds the ratio to it
    // (1 on every body row: no product there); the Rx window is divided by its flat value (a common factor of the
    // received signal cancels in the pilot equaliser) and rows 1..13 of the Rx gather skip the product
    // (BerParams::flat_tx / flat_rx: bit v = window pair v)
    for (int vv = 0; vv < nvar; ++vv) {
        const T* gw = reinterpret_cast<const T*>(prm.win_tx) + (size_t)vv * n_tx;
        const T* gr = reinterpret_cast<const T*>(prm.win_rx) + (size_t)vv * (N + prm.tail_rx);
        const bool ft = (prm.flat_tx >> vv) & 1, fr = (prm.flat_rx >> vv) & 1;
        const T wflat = ft ? gw[beta] : (T)1, rflat = fr ? gr[prm.tail_rx] : (T)1;
        for (int i = tid; i < n_tx; i += NT) wtx_all[vv * WTXL + i] = ft ? gw[i] / wflat : gw[i] * TCV_XSCALE;
        for (int i = tid; i < N + prm.tail_rx; i += NT) wrx_all[vv * WRXL + i] = gr[i] / rflat;
    }
    // constellation table of window pair vv for the Tx stage
    auto build_qtx = [&](int vv) {
        const bool ft = (prm.flat_tx >> vv) & 1;
        const T wflat = ft ? reinterpret_cast<const T*>(prm.win_tx)[(size_t)vv * n_tx + beta] : (T)1;
        for (int i = tid; i < (1 << prm.bits); i += NT) {
            const C2 q = mk2<T>((T)(2 * (i >> hb) - (m - 1)), (T)(2 * (i & (m - 1)) - (m - 1)));
            qtx[i] = ft ? cscale(wflat * TCV_XSCALE, q) : q;
        }
    };
    for (int i = tid; i < PAD; i += NT) ahi[i] = 0u;
    for (int i = tid; i < 2 * TBL / 4; i += NT) reinterpret_cast<uint32_t*>(bt + 2 * TBL)[i] = 0u;   // (B0, B1: their rows 4..7 stay zero)
    for (int i = tid; i < (1 << prm.bits); i += NT) qlut[i] = mk2<T>((T)(2 * (i >> hb) - (m - 1)), (T)(2 * (i & (m - 1)) - (m - 1)));
    build_qtx(0);
    if (tid == 0 && prm.bits < 8) { qlut[255] = mk2<T>(0, 0); qtx[255] = mk2<T>(0, 0); }
    const uint32_t gxm = gray_xor_mask(prm.bits, prm.constellation);
    uint32_t* const racc = reinterpret_cast<uint32_t*>(smem_raw + lay.off_res);   // RES: [nvar][N][2] = {bit, sym}
    if constexpr (RES) { for (int i = tid; i < 2 * N * nvar; i += NT) racc[i] = 0u; }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    if (!HS && prm.guard > 0) {
        const unsigned d0 = slice_index(mk2<T>(0, 0), hb);
        for (int tt = tid; tt < TPF; tt += NT) {
            uint32_t ff[4] = {0, 0, 0, 0}, dd[4] = {0, 0, 0, 0};
            for (int q = 0; q < 16; ++q)
                if (!bin_active<N>(tt + q * TPF, prm.guard)) { ff[q >> 2] |= 0xffu << (8 * (q & 3)); dd[q >> 2] |= d0 << (8 * (q & 3)); }
            gmask[2 * tt] = make_uint4(ff[0], ff[1], ff[2], ff[3]);
            gmask[2 * tt + 1] = make_uint4(dd[0], dd[1], dd[2], dd[3]);
        }
        __syncthreads();
    }

    // this thread's operand row inside every tile (TMEM lane) and its half of the row's four outputs
    const int wg = (warp >> 2) & 1, row = (warp & 3) * 32 + lane;
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);      // the warp index as a value the compiler knows to be warp-uniform
    const int tp = TG == 1 ? 0 : (warp_u >> 3);                // this warp's tile set: tiles tp, tp + TG, ...
    const uint32_t tlane = tmem + ((uint32_t)((warp_u & 3) * 32) << 16) + (uint32_t)(8 * ((warp_u >> 2) & 1));
    uint32_t phase = 0;
    constexpr bool MMAW = tconv2_mma_warp_threads(N, NT) > 0;       // a dedicated MMA warp (warp NW)
    constexpr int NTB = NT + tconv2_mma_warp_threads(N, NT);        // threads that meet at the "stream complete" barrier
    // MMA descriptors of tile 0, K step 0 (tile: +2048 B = +128 in the address field, K step: +32 B = +2; B operand: +256 B = +16)
    const uint64_t d_ahi = tcv_desc(tcv_smem_u32(ahi), 16, 128), d_alo = tcv_desc(tcv_smem_u32(alo), 16, 128);
    // Taps operand (16 columns = two core matrices of 8 rows, TBL bytes apart): the accumulator columns a thread reads are kept
    // together -- column 8 g + r (g = output pair, r = 2 (o & 1) + comp) takes hi.T_hi + lo.T_hi and column 8 g + 4 + r the
    // correction hi.T_lo, so one tcgen05.ld.x8 fetches a thread's two outputs with their corrections.  Blocks A_g (hi
    // stream: rows 0..3 = T_hi, rows 4..7 = T_lo of pair g) and B_g (lo stream: rows 0..3 = T_hi, rows 4..7 = zeros).
    const uint64_t d_bhl = tcv_desc(tcv_smem_u32(bt), 128, TBL), d_bh0 = tcv_desc(tcv_smem_u32(bt + 2 * TBL), 128, TBL);
    // channel output r, parked over the dead split stream in two halves: R[wg] holds outputs 2 wg, 2 wg + 1 of every operand
    // row as one 16-byte chunk per row -- consecutive lanes store consecutive chunks (no bank conflicts) and a receiver
    // thread's samples i = i0 + q TPF all have the same i mod 4, i.e. the same half and chunk slot: base + immediate
    const int RCH = NTILE * 128 + 4;            // chunks per half (+4: the halves sit 64 bytes apart modulo 128)
    // extras of the noise draws (ber_kernel.cuh: noise_draw48)
    const N48Geom ng = n48_geom(prm);
    const int xt = (t - ng.base) & (TPF - 1);   // this thread's extras: x = xt + lev * TPF

    // distributed shared memory: the previous CTA's split stream (its last Tx tail and the convolution history)
    const uint32_t* prev_uh = uh;
    const uint32_t* prev_ul = ul;
    if constexpr (CL > 1) {
        if (rank > 0) {
            prev_uh = cooperative_groups::this_cluster().map_shared_rank(uh, rank - 1);
            prev_ul = cooperative_groups::this_cluster().map_shared_rank(ul, rank - 1);
        }
    }
    const long long fslot = blockIdx.x / CL, nslots = gridDim.x / CL;   // frames in flight on the grid
#if TCV2_TRACE
    __shared__ long long trace_buf[17 * 12];
    int trace_it = 0;
#endif
    if (MMAW && warp >= NW) {
        if constexpr (tconv2_setmaxnreg(N, NT)) asm volatile("setmaxnreg.dec.sync.aligned.u32 24;" ::: "memory");
        // ===== the MMA warp: the CTA's extra warp issues every tcgen05.mma of the kernel and nothing else =====
        // An issuing thread sits in front of the tensor core's short queue for as long as the convolution takes (~40 cycles per
        // MMA, bound by the operand reads: ~2200 cycles per frame at N = 256).  Measured with the issue spread over four of
        // the eight working warps: those four reached the power barrier ~1900 cycles after the others, every frame.  Here
        // the working warps only announce their stores (bar.arrive) and draw their noise while this warp waits for the
        // stream (bar.sync), issues, and otherwise just keeps the CTA's / cluster's barrier sequence.
        for (long long j = fslot; j < prm.n_frames; j += nslots) {
            for (int var = 0; var < nvar; ++var) {
#if TCV2_TRACE
                const bool trace_on = blockIdx.x == 0 && trace_it >= 3 && trace_it < 6;
                ++trace_it;
                TCV2_STAMP(0);
#endif
                frame_sync<CL>();                                         // Tx: every symbol's tail is in place
                TCV2_STAMP(1);
                if constexpr (CL > 1) asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
                if (TCV2_DEBUG_BARRIERS) __syncthreads();
                else asm volatile("bar.sync %0, %1;" :: "n"(TCV2_BAR_STREAM), "n"(NTB) : "memory");   // the split stream is complete
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                TCV2_STAMP(2);
                if (warp_u == NW && tcv_elect_one()) {
#pragma unroll
                    for (int ti = 0; ti < NTILE; ++ti) {
                        const uint32_t tacc = tmem + (uint32_t)(16 * ti);
#pragma unroll
                        for (int k = 0; k < KS; ++k) {
                            tcv_mma(tacc, d_ahi + (uint64_t)(ti * 128 + k * 2), d_bhl + (uint64_t)(k * 16), k != 0);
                            tcv_mma(tacc, d_alo + (uint64_t)(ti * 128 + k * 2), d_bh0 + (uint64_t)(k * 16), 1u);
                        }
                        // completes when all MMAs issued so far have
#pragma unroll
                        for (int sgm = 0; sgm < NSEG; ++sgm)
                            if (ti == (tconv2_seg_end(NSEG, NTILE, sgm) < NTILE - 1 ? tconv2_seg_end(NSEG, NTILE, sgm) : NTILE - 1))
                                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(tcv_smem_u32(bar + sgm)) : "memory");
                    }
                }
                __syncwarp();
                TCV2_STAMP(3);
#if TCV2_TRACE
                if (trace_on) { tcv_mbar_wait(tcv_smem_u32(bar + NSEG - 1), phase); TCV2_STAMP(4); }
                phase ^= 1u;
#endif
                if constexpr (CL > 1) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
                frame_sync<CL>();                                         // power partials
                if (rank == 0) __syncthreads();                           // pilot published
                frame_sync<CL>();                                         // equaliser taps
#if TCV2_TRACE
                if (trace_on) { __syncthreads(); __syncthreads(); }
#endif
                if (TCV2_DEBUG_BARRIERS) frame_sync<CL>();
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        frame_sync<CL>();
        return;
    }
    if constexpr (MMAW && tconv2_setmaxnreg(N, NT)) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" :: "n"(tconv2_work_regs(NT)) : "memory");
    long long f = prm.frame_begin + fslot * prm.frame_step;
    const long long df = nslots * prm.frame_step;
    long long fe = 0, de = 0;
    int ci = 0, si = 0, dc = 0, ds = 0;
    if constexpr (!VERIFY) {
        const long long q = f / prm.ensemble, dq = df / prm.ensemble;
        fe = f - q * prm.ensemble;   de = df - dq * prm.ensemble;
        si = (int)(q / prm.C);       ci = (int)(q - (long long)si * prm.C);
        ds = (int)(dq / prm.C);      dc = (int)(dq - (long long)ds * prm.C);
    }
    // RES with a segment table: f above is the local index g, every frame's (f, si, ci) comes from seg_frame (ber_kernel.cuh);
    // the CTAs of a cluster share fslot, so they map the same g
    [[maybe_unused]] long long g = f;
    if constexpr (RES) { if (prm.seg) seg_frame(prm, g, f, si, ci); }
    // RES: cells of the counters and this CTA's current one
    const size_t ncell = RES ? (size_t)prm.n_snr * (prm.res_chan ? prm.C : 1) : 0;
    int rcell = RES ? (prm.res_chan ? si * prm.C + ci : si) : 0;
    unsigned rfr = 0;
    const unsigned rlim = RES ? res_frame_limit(prm.S, prm.bits) : 0u;
    for (long long j = fslot; j < prm.n_frames; j += nslots) {
#if TCV2_TRACE
        const bool trace_on = blockIdx.x == 0 && trace_it >= 3 && trace_it < 6;
        ++trace_it;
        TCV2_STAMP(0);
#endif
        if constexpr (VERIFY) { ci = (int)f; si = (int)f; }
        const T snr_lin = reinterpret_cast<const T*>(prm.snr_lin)[si];
      // every window pair of the plan on this frame's symbols (drawn once), each with its own noise stream
      // (wofdm_simulation.py:183-236: optimised and RC windows on one signal_digmod; main_BER_calculation.m:118-198)
      for (int var = 0; var < nvar; ++var) {
        const bool flat_tx = HS || ((prm.flat_tx >> var) & 1), flat_rx = (prm.flat_rx >> var) & 1;
        const T* const wtx = wtx_all + var * WTXL;
        const T* const wrx = wrx_all + var * WRXL;
        // ---- taps operand of this frame: n = 2o + comp (o < 4), K pair jj = sample offset in the row, tap l = LB-1 + o - jj
        auto build_tap = [&](int e) {
            // (a warp covers one 16-byte K chunk of all 8 rows: its stores spread over the banks)
            const int n = (e >> 2) & 7, jj = (e >> 5) * 4 + (e & 3);
            const int o = n >> 1, l = PAD + o - jj;
            C2 tpv = mk2<T>(0, 0);
            if (l >= 0 && l < L) tpv = reinterpret_cast<const C2*>(prm.chan)[(size_t)ci * L + l];
            tpv = cscale(TCV_HSCALE, tpv);
            const C2 v = (n & 1) ? mk2<T>(tpv.y, tpv.x) : mk2<T>(tpv.x, -tpv.y);     // multiplies (Re u, Im u)
            uint32_t hi, lo;
            split_h2(v, hi, lo);
            const int off = (n >> 2) * TBL + (jj >> 2) * 128 + (n & 3) * 16 + (jj & 3) * 4;
            *reinterpret_cast<uint32_t*>(bt + off) = hi;
            *reinterpret_cast<uint32_t*>(bt + off + 64) = lo;
            *reinterpret_cast<uint32_t*>(bt + 2 * TBL + off) = hi;
        };
        constexpr int NTAP = 8 * (PAD + 4);
        if constexpr (NTAP + PAD + ZERO <= NT) {                             // (LB = 21) one element per thread
            if (tid < NTAP) {
                if (var == 0) build_tap(tid);
            } else if (tid < NTAP + PAD) {
                alo[tid - NTAP] = 0u;                                        // (r of the previous frame lay over it)
            } else if (tid - (NTAP + PAD) < ZERO) {
                const int i = body + tid - (NTAP + PAD);                     // the linear convolution sees zeros behind the stream
                uh[i] = 0u; ul[i] = 0u;
            }
        } else {
            if (var == 0)
                for (int e = tid; e < NTAP; e += NT) build_tap(e);
            for (int e = NT - 1 - tid; e < PAD + ZERO; e += NT) {           // (the last threads: the first ones build the taps)
                if (e < PAD) alo[e] = 0u;
                else { const int i = body + e - PAD; uh[i] = 0u; ul[i] = 0u; }
            }
        }

        // =========================== transmitter ===========================
        if (!HS && prm.tx_stream != nullptr) {          // uniform: masked Tx stream from tx_mask_kernel (mask_kernel.cuh)
            for (int e = tid; e < S * TPF; e += NT) {
                const int tt = e % TPF;
                uint32_t w[4];
                load_sym_idx<N, VERIFY>(prm, f, sb + e / TPF, tt, w);
                if (prm.guard > 0) {
                    const uint4 gf = gmask[2 * tt], gd = gmask[2 * tt + 1];
                    w[0] = (w[0] & ~gf.x) | gd.x; w[1] = (w[1] & ~gf.y) | gd.y;
                    w[2] = (w[2] & ~gf.z) | gd.z; w[3] = (w[3] & ~gf.w) | gd.w;
                }
                symw[e] = make_uint4(w[0], w[1], w[2], w[3]);
            }
            if constexpr (TXY) {             // (its own instantiations: the production kernels stay as they are)
                // the frame this CTA takes next: its S columns of Y are contiguous -- one bulk prefetch into L2 (the loader is
                // bound by the latency of its gather, and the product wrote Y through to HBM)
                if (tid == 0 && j + nslots < prm.n_frames)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(prm.tx_y + (size_t)(j + nslots) * S * prm.tx_yp),
                                 "r"((uint32_t)(S * prm.tx_yp * 4)) : "memory");
                tconv2_load_masked<NT>(prm.tx_y + (size_t)j * S * prm.tx_yp, prm.tx_yp, S, stride, n_tx, body, uh, ul, tid);
            } else {
                const float2* src = prm.tx_stream + (size_t)j * body;
                for (int i = tid; i < body; i += NT) {
                    uint32_t hi, lo;
                    split_h2(cscale(TCV_XSCALE, src[i]), hi, lo);
                    uh[i] = hi; ul[i] = lo;
                }
            }
            frame_sync<CL>();
        } else {
            const bool act = slot < S;
            const int s = TCV2_SLOT_SYMBOL(slot, S);
            const int se = act ? s : S - 1;     // idle slots shadow the last symbol (identical stores)
            const bool first = sb + se == 0;    // the frame's first symbol has no predecessor
            C2 v[16];
            {
                uint32_t w[4], wq[4];
                if (var == 0) {
                    load_sym_idx<N, VERIFY>(prm, f, sb + se, t, w);
                } else {                           // the symbols of the frame, as stored by the first window pair
                    const uint4 ws = symw[se * TPF + t];
                    w[0] = ws.x; w[1] = ws.y; w[2] = ws.z; w[3] = ws.w;
                }
#pragma unroll
                for (int jw = 0; jw < 4; ++jw) wq[jw] = w[jw];
                if (!HS && prm.guard > 0) {
                    const uint4 gf = gmask[2 * t], gd = gmask[2 * t + 1];
                    const uint32_t ff[4] = {gf.x, gf.y, gf.z, gf.w}, dd[4] = {gd.x, gd.y, gd.z, gd.w};
#pragma unroll
                    for (int jw = 0; jw < 4; ++jw) { wq[jw] = w[jw] | ff[jw]; w[jw] = (w[jw] & ~ff[jw]) | dd[jw]; }
                }
                if (var == 0) symw[se * TPF + t] = make_uint4(w[0], w[1], w[2], w[3]);
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = qtx[sym_byte(wq, q)];
            }
            fft_regs<T, N, +1, FPP>(v, t, xb, tw, slot);
            // CP/CS insertion + Tx window (transmitter.py:13-35, 61-87); heads i < tail_tx overlap the previous symbol's
            // falling tail (wofdm_simulation.py:190-203) and are added after the barrier
            uint32_t* const sh = uh + se * stride;
            uint32_t* const sl = ul + se * stride;
            if (flat_tx) {                        // uniform (implies cp, cs >= tail_tx: the body lies in the flat part)
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    uint32_t hi, lo;
                    split_h2(v[q], hi, lo);
                    sh[t + q * TPF + cp] = hi; sl[t + q * TPF + cp] = lo;
                }
            } else if (cp >= beta) {
                T wv[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) wv[q] = wtx[t + q * TPF + cp];
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    uint32_t hi, lo;
                    split_h2(cscale(wv[q], v[q]), hi, lo);
                    sh[t + q * TPF + cp] = hi; sl[t + q * TPF + cp] = lo;
                }
            } else {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int i = t + q * TPF + cp;
                    if (q >= ER || i >= beta || first) {
                        uint32_t hi, lo;
                        split_h2(cscale(wtx[i], v[q]), hi, lo);
                        sh[i] = hi; sl[i] = lo;
                    }
                }
            }
#pragma unroll
            for (int q = 16 - ER; q < 16; ++q) {
                if (q * TPF + TPF > N - cp) {             // uniform: this register row reaches the prefix
                    const int i = t + q * TPF - (N - cp);
                    if (i >= 0 && (i >= beta || first)) {
                        uint32_t hi, lo;
                        split_h2(cscale(wtx[i], v[q]), hi, lo);
                        sh[i] = hi; sl[i] = lo;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < ER; ++q) {
                if (q * TPF < cs) {                        // uniform: ... the suffix
                    const int i = t + q * TPF + cp + N;
                    if (i < n_tx) {
                        uint32_t hi, lo;
                        split_h2(cscale(wtx[i], v[q]), hi, lo);
                        sh[i] = hi; sl[i] = lo;
                    }
                }
            }
            TCV2_STAMP(1);
            frame_sync<CL>();                   // every symbol's tail is in place
            TCV2_STAMP(2);
            // the falling tail of the previous symbol: same buffer, or the previous CTA's (behind its kept samples)
            const uint32_t* const th = (CL > 1 && se == 0) ? prev_uh + sec : sh;
            const uint32_t* const tl = (CL > 1 && se == 0) ? prev_ul + sec : sl;
            if (beta > 0 && act && !first) {
#pragma unroll
                for (int q = 16 - ER; q < 16; ++q) {
                    if (q * TPF + TPF > N - cp) {
                        const int i = t + q * TPF - (N - cp);
                        if (i >= 0 && i < beta) {
                            uint32_t hi, lo;
                            split_h2(caxpy(wtx[i], v[q], join_h2(th[i], tl[i])), hi, lo);
                            sh[i] = hi; sl[i] = lo;
                        }
                    }
                }
                if (!HS && cp < beta) {
#pragma unroll
                    for (int q = 0; q < ER; ++q) {
                        const int i = t + q * TPF + cp;
                        if (i < beta) {
                            uint32_t hi, lo;
                            split_h2(caxpy(wtx[i], v[q], join_h2(th[i], tl[i])), hi, lo);
                            sh[i] = hi; sl[i] = lo;
                        }
                    }
                }
            }
        }
        if constexpr (CL > 1) {
            // convolution history: the last PAD stream samples of the previous CTA (none of them is a head)
            if (rank > 0 && tid < PAD) { ahi[tid] = prev_uh[sec - PAD + tid]; alo[tid] = prev_ul[sec - PAD + tid]; }
            // "I have taken what I need from my neighbour's stream": awaited before anybody parks r over a stream
            asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
        }
        TCV2_STAMP(3);
        // the tensor core reads shared memory through the async proxy
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");

        // =========================== channel + AWGN ===========================
        // r = conv(h, u) (wofdm_simulation.py:206-209) on the tensor cores; y = r + sqrt(Pr*10^(-snr/10)/Pn) n with Pr, Pn
        // summed over the whole frame (:135-138; noise_norm 1: over the full convolution, main_BER_calculation.m:260-261,289-292)
        // The MMA warp (above) waits for the whole stream and issues the frame's MMAs; the working warps only announce their
        // stores and go on to the noise draws.  Without an MMA warp (NT = 512), TCV2_NISSUE working warps do its job first.
        // The issuing warps rotate from frame to frame.  The rotation is keyed on the frame's global id and its noise stream
        // (variant + var), never on the CTA or on the frames it decided before: the accumulator pass below hands the issuers'
        // tiles to other warps, so it sets the association of the frame-power sum, and a frame's counters must not depend on
        // where it runs (shards, segments, devices, a pair alone).  The id is hashed (Fibonacci): a CTA's frames lie
        // nslots * frame_step apart, often a multiple of 16, which would freeze a rotation by f itself.  (The shuffle keeps the
        // key and what derives from it in vector registers, as the CTA index was: computed in the uniform datapath the same key
        // cost 3 % at configs[4], and so did a fixed key -- tools/bench_ber_n1024_rotation.py.  With an MMA warp nobody reads it.)
        const uint32_t issuer = MMAW ? 0u : __shfl_sync(0xffffffffu, ((uint32_t)f * 0x9E3779B9u >> 28) + prm.variant + (uint32_t)(var + rank), 0);
        const int irank = (int)(((uint32_t)warp_u - issuer) & (NW - 1));   // warp-uniform: issuing warps have irank < TCV2_NISSUE
        const bool is_issuer = !MMAW && irank < TCV2_NISSUE;
        constexpr bool STAG = !MMAW && TCV2_STAGGER && !TCV2_DEBUG_BARRIERS;
        const int igrp = irank >> 2;                                    // staggered issue: this warp's group
        auto issue_group = [&](auto gc) {                               // group g's quarter of the tiles, shared round-robin by its four warps
            constexpr int g = decltype(gc)::value;
            (void)g;
            if constexpr (STAG) {
                if (igrp == g) {
                    asm volatile("bar.sync %0, %1;" :: "n"(TCV2_BAR_STREAM - g), "n"(NTB) : "memory");
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (tcv_elect_one()) {
                        constexpr int g0 = NTILE * g / 4, g1 = NTILE * (g + 1) / 4;
#pragma unroll
                        for (int ti = g0; ti < g1; ++ti) {
                            if (((ti - g0) & 3) == (irank & 3)) {
                                const uint32_t tacc = tmem + (uint32_t)(16 * ti);
#pragma unroll
                                for (int k = 0; k < KS; ++k) {
                                    tcv_mma(tacc, d_ahi + (uint64_t)(ti * 128 + k * 2), d_bhl + (uint64_t)(k * 16), k != 0);
                                    tcv_mma(tacc, d_alo + (uint64_t)(ti * 128 + k * 2), d_bh0 + (uint64_t)(k * 16), 1u);
                                }
                            }
                        }
                        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(tcv_smem_u32(bar)) : "memory");
                    }
                    __syncwarp();
                }
            }
        };
        if constexpr (STAG) {
            static_assert(NW == 16 && NSEG == 1, "four groups of four warps, one commit per warp");
            // "my part of the stream is stored" to the three groups this warp is not in
            if (igrp != 0) asm volatile("bar.arrive %0, %1;" :: "n"(TCV2_BAR_STREAM), "n"(NTB) : "memory");
            if (igrp != 1) asm volatile("bar.arrive %0, %1;" :: "n"(TCV2_BAR_STREAM - 1), "n"(NTB) : "memory");
            if (igrp != 2) asm volatile("bar.arrive %0, %1;" :: "n"(TCV2_BAR_STREAM - 2), "n"(NTB) : "memory");
            if (igrp != 3) asm volatile("bar.arrive %0, %1;" :: "n"(TCV2_BAR_STREAM - 3), "n"(NTB) : "memory");
            issue_group(std::integral_constant<int, 0>{});
        }
        if (TCV2_DEBUG_BARRIERS) __syncthreads();
        if (STAG) {
        } else if (is_issuer) {
            if (!TCV2_DEBUG_BARRIERS) asm volatile("bar.sync %0, %1;" :: "n"(TCV2_BAR_STREAM), "n"(NTB) : "memory");
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (tcv_elect_one()) {
#pragma unroll
                for (int ti = 0; ti < NTILE; ++ti) {
                    if (ti % TCV2_NISSUE == irank) {                      // the issuing warps share the tiles round-robin
                        const uint32_t tacc = tmem + (uint32_t)(16 * ti);
#pragma unroll
                        for (int k = 0; k < KS; ++k) {
                            tcv_mma(tacc, d_ahi + (uint64_t)(ti * 128 + k * 2), d_bhl + (uint64_t)(k * 16), k != 0);
                            tcv_mma(tacc, d_alo + (uint64_t)(ti * 128 + k * 2), d_bh0 + (uint64_t)(k * 16), 1u);
                        }
                    }
#pragma unroll
                    for (int sgm = 0; sgm < NSEG; ++sgm)
                        if (ti == (tconv2_seg_end(NSEG, NTILE, sgm) < NTILE - 1 ? tconv2_seg_end(NSEG, NTILE, sgm) : NTILE - 1))
                            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(tcv_smem_u32(bar + sgm)) : "memory");
                }
            }
            __syncwarp();
        } else if (!TCV2_DEBUG_BARRIERS) {
            asm volatile("bar.arrive %0, %1;" :: "n"(TCV2_BAR_STREAM), "n"(NTB) : "memory");
        }
        TCV2_STAMP(4);
        // ---- noise, in receiver layout and in registers (ber_kernel.cuh: noise_draw48): the 16 samples this thread's FFT
        //      rows gather, and its extras; |n|^2 partial
        // (only the extras of levels 0 and 1 can be overlap-add samples the receiver gathers, tail_rx / 2 <= TPF; the others
        //  count in the noise power and are dropped)
        C2 nz[16], nx[2];
        C2 pr2 = mk2<T>(0, 0), pn2 = mk2<T>(0, 0), pnx = mk2<T>(0, 0);
        // HS: the draws are register arithmetic only, and with the switches as constants ptxas hoists most of them above the
        // bar.arrive above (468 SASS instructions between the Tx barrier and the arrive instead of 112): the MMA warp then waits
        // for every working warp's draws before it issues, and the accumulator pass waits for the MMAs.  So there the draws key
        // on a frame id that passes through a shared-memory load behind the arrive (ahi[0], the operand's zero pad: always 0),
        // which ptxas does not move across the barrier.
        long long fn = f;
        if constexpr (HS) {
            static_assert(CL == 1, "ahi[0] is zero only with one CTA per frame: a CTA of rank > 0 writes its neighbour's history there");
            uint32_t z;
            asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(z) : "r"(tcv_smem_u32(ahi)) : "memory");
            fn += z;
        }
        {
            const bool act = slot < S;
            const int se = act ? TCV2_SLOT_SYMBOL(slot, S) : S - 1;
            const int sg = sb + se;                                      // symbol index in the frame
            const int xas = ng.xa + (sg == prm.S - 1 ? ng.tailx : 0);    // extras of this symbol (uniform per transform group)
            const int nlev = (xas + TPF - 1) / TPF;
            const int pbase = sg * stride;
            if constexpr (VERIFY) {
                const double2* nin = prm.noise_in + (size_t)f * prm.noise_len + pbase;
#pragma unroll
                for (int q = 0; q < 16; ++q) nz[q] = to_v2<T>(nin[prm.rm + hh + ((t + q * TPF + prm.shift) & (N - 1))]);
#pragma unroll
                for (int lev = 0; lev < N48_MAXLEV; ++lev) {
                    const int x = xt + lev * TPF;
                    const C2 e = x < xas ? to_v2<T>(nin[n48_extra_offset(prm, ng, x)]) : mk2<T>(0, 0);
                    if (lev < 2) nx[lev] = e; else pnx = csq_acc(e, pnx);
                }
            } else {
                const uint32_t q0 = (uint32_t)(sg * TPF + t) * (uint32_t)N48_CALLS;
#pragma unroll
                for (int gq = 0; gq < 2; ++gq) {
                    const uint4 ca = noise48_call(prm, fn, q0 + 3 * gq, var), cb = noise48_call(prm, fn, q0 + 3 * gq + 1, var);
                    const uint4 cc = noise48_call(prm, fn, q0 + 3 * gq + 2, var);
                    gauss_quad48(ca.x, ca.y, cc.x, nz[8 * gq + 0], nz[8 * gq + 1]);
                    gauss_quad48(ca.z, ca.w, cc.y, nz[8 * gq + 2], nz[8 * gq + 3]);
                    gauss_quad48(cb.x, cb.y, cc.z, nz[8 * gq + 4], nz[8 * gq + 5]);
                    gauss_quad48(cb.z, cb.w, cc.w, nz[8 * gq + 6], nz[8 * gq + 7]);
                    if (gq == 0) issue_group(std::integral_constant<int, 1>{}); else issue_group(std::integral_constant<int, 2>{});
                }
                nx[0] = nx[1] = mk2<T>(0, 0);
                if (nlev > 0) {                                          // uniform per transform group
                    const uint4 c6 = noise48_call(prm, fn, q0 + 6, var);
                    gauss_quad48(c6.y, c6.z, c6.x, nx[0], nx[1]);
                    if (xt >= xas) nx[0] = mk2<T>(0, 0);
                    if (xt + TPF >= xas) nx[1] = mk2<T>(0, 0);
                    // further level pairs (long prefixes; the last symbol under MATLAB's full-convolution sums): rare, out of line
                    if constexpr (LB > TCV_LB) {
                        if (nlev > 2) pnx = n48_more_extras(prm, fn, q0, var, nlev, xt, TPF, xas);
                    } else if (nlev > 2) {                               // (at most N48_MAXLEV_SHORT = 6 levels: ber_host.cu)
                        const uint4 c7 = noise48_call(prm, fn, q0 + 7, var);
                        C2 e2, e3;
                        gauss_quad48(c7.x, c7.y, c6.w, e2, e3);
                        if (xt + 2 * TPF < xas) pnx = csq_acc(e2, pnx);
                        if (xt + 3 * TPF < xas) pnx = csq_acc(e3, pnx);
                        if (nlev > 4) {
                            const uint4 c8 = noise48_call(prm, fn, q0 + 8, var);
                            gauss_quad48(c7.w, c8.x, c7.z, e2, e3);
                            if (xt + 4 * TPF < xas) pnx = csq_acc(e2, pnx);
                            if (xt + 5 * TPF < xas) pnx = csq_acc(e3, pnx);
                        }
                    }
                }
            }
            if constexpr (VERIFY) { issue_group(std::integral_constant<int, 1>{}); issue_group(std::integral_constant<int, 2>{}); }
            issue_group(std::integral_constant<int, 3>{});
            if (act) {
#pragma unroll
                for (int q = 0; q < 16; ++q) pn2 = csq_acc(nz[q], pn2);
                pn2 = csq_acc(nx[0], pn2);
                pn2 = csq_acc(nx[1], pn2);
                pn2 = cadd(pn2, pnx);
            }
        }
        TCV2_STAMP(5);
        // ---- the channel output, once: frame-wide signal power, r parked over the dead split stream
        int seg_waited = 0;                        // (compile-time in the unrolled passes below)
        auto wait_tiles = [&](int tmax) {          // tiles 0..tmax are complete (and nobody reads their stream any more)
            const int k = tconv2_seg_of(NSEG, NTILE, tmax < NTILE - 1 ? tmax : NTILE - 1);
            for (; seg_waited <= k; ++seg_waited) tcv_mbar_wait(tcv_smem_u32(bar + seg_waited), phase);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        };
        wait_tiles(0);
        TCV2_STAMP(6);
        if constexpr (CL > 1) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
        constexpr int GT = TCV2_GT;                // tiles per batch of accumulator loads (one wait per batch)
        if constexpr (!MMAW && TCV2_REBALANCE && !STAG) {
            // The working warps issue the MMAs (N = 1024): the four issuing warps of this frame reach this point ~2000 cycles
            // after the others (phase traces: they sat in front of the tensor core's queue), and everybody would wait for
            // them at the power barrier.  So they skip this pass: the tiles of a tensor-memory lane quarter -- which only the
            // four warps w = quarter (mod 4) can read -- go to the three warps of the quarter that did not issue (exactly one
            // did: the issuers are four consecutive warps), all 16 columns of a row in one tcgen05.ld.x16.
            static_assert(NW == 16, "four warps per tensor-memory lane quarter");
            if (!is_issuer) {
                const int wi = (int)((issuer + (((uint32_t)warp_u - issuer) & 3u)) & (NW - 1));   // the quarter's issuing warp
                const int k = warp_u >> 2, ki = wi >> 2;
                const int r3 = k - (k > ki ? 1 : 0);                               // my rank among the quarter's three others
                const uint32_t tq = tmem + ((uint32_t)((warp_u & 3) * 32) << 16);
                float4* const rq = reinterpret_cast<float4*>(rb) + row;
                constexpr int NPW = (NTILE + 2) / 3;                                // tiles per warp
                constexpr int GR = 2;                                               // tiles per batch of loads
#pragma unroll
                for (int i0 = 0; i0 < NPW; i0 += GR) {
                    C2 c[GR][8];
                    wait_tiles(3 * (i0 + GR - 1) + 2);
#pragma unroll
                    for (int u = 0; u < GR; ++u)
                        if (i0 + u < NPW) tcv_ld16(tq + (uint32_t)(16 * min(3 * (i0 + u) + r3, NTILE - 1)), c[u]);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int u = 0; u < GR; ++u) {
                        if (i0 + u < NPW) {
                            const int tt = 3 * (i0 + u) + r3, p = 512 * tt + 4 * row;
                            if (tt < NTILE) {
#pragma unroll
                                for (int wq = 0; wq < 2; ++wq) {
                                    const C2 r0 = cadd(c[u][4 * wq], c[u][4 * wq + 2]), r1 = cadd(c[u][4 * wq + 1], c[u][4 * wq + 3]);
                                    if (p + 2 * wq < npow) pr2 = csq_acc(r0, pr2);
                                    if (p + 2 * wq + 1 < npow) pr2 = csq_acc(r1, pr2);
                                    if (p + 2 * wq < sec) rq[wq * RCH + 128 * tt] = make_float4(r0.x, r0.y, r1.x, r1.y);   // (a sample past the frame is never gathered)
                                }
                            }
                        }
                    }
                }
            }
        } else {
        float4* const rst = reinterpret_cast<float4*>(rb) + wg * RCH + row;
#pragma unroll
        for (int t0 = 0; t0 < NTH; t0 += GT) {
            C2 a0[GT], a1[GT], b0[GT], b1[GT];
            wait_tiles(TG * (t0 + GT - 1) + TG - 1);
#pragma unroll
            for (int u = 0; u < GT; ++u) {
                if (t0 + u < NTH) {
                    const int tt = min(TG * (t0 + u) + tp, NTILE - 1);      // (a set's tile past the frame: result masked below)
                    if constexpr (N == 512) {        // (register bound: an x8 load's eight consecutive registers cost spills there)
                        tcv_ld4(tlane + (uint32_t)(16 * tt), a0[u], a1[u]);
                        tcv_ld4(tlane + (uint32_t)(16 * tt + 4), b0[u], b1[u]);
                    } else {
                        tcv_ld8(tlane + (uint32_t)(16 * tt), a0[u], a1[u], b0[u], b1[u]);
                    }
                }
            }
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int u = 0; u < GT; ++u) {
                if (t0 + u < NTH) {
                    const int tt = TG * (t0 + u) + tp, p = 512 * tt + 4 * row + 2 * wg;
                    const C2 r0 = cadd(a0[u], b0[u]), r1 = cadd(a1[u], b1[u]);
                    if (tt < NTILE - 2) {
                        pr2 = csq_acc(r0, pr2);
                        pr2 = csq_acc(r1, pr2);
                        rst[128 * tt] = make_float4(r0.x, r0.y, r1.x, r1.y);
                    } else if (tt < NTILE) {
                        if (p < npow) pr2 = csq_acc(r0, pr2);
                        if (p + 1 < npow) pr2 = csq_acc(r1, pr2);
                        if (p < sec) rst[128 * tt] = make_float4(r0.x, r0.y, r1.x, r1.y);   // (a sample past the frame is never gathered)
                    }
                }
            }
        }
        }
        phase ^= 1u;
        T pr = warp_sum(pr2.x + pr2.y), pn = warp_sum(pn2.x + pn2.y);
        if (lane == 0) {
            // warp partials go to slot rank*NW + warp of EVERY CTA of the frame: same order, same gain everywhere
#pragma unroll
            for (int r = 0; r < CL; ++r) {
                T* rr = red;
                if constexpr (CL > 1) rr = cooperative_groups::this_cluster().map_shared_rank(red, r);
                rr[rank * NW + warp] = pr; rr[32 + rank * NW + warp] = pn;
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        TCV2_STAMP(7);
        frame_sync<CL>();                          // r and the power partials are complete
        TCV2_STAMP(8);
        const T g = noise_gain(block_total<CL * NW>(red), snr_lin, block_total<CL * NW>(red + 32));

        // =========================== receiver ===========================
        // block s: y = r + g n; z[k] = wrx[k]*y[s*stride + rm + k]; o[n] = sum_{k = n + hh (mod N)} z[k];
        // q[n] = o[(n + shift) mod N]; Y = DFT(q)   (receiver.py:13-133)
        unsigned bit_cnt = 0, sym_cnt = 0;
        {
            const bool act = slot < S;
            const int s = TCV2_SLOT_SYMBOL(slot, S);
            const int se = act ? s : S - 1;
            C2 v[16];
            // r of stream sample i: half (i >> 1) & 1, chunk i >> 2, element i & 1 -- constant i mod 4 for all of this thread's samples
            const int ib = se * stride + prm.rm + hh;                    // stream position of block offset n = 0
            const int i0 = ib + t + prm.shift;
            const C2* const rsel = rb + ((i0 >> 1) & 1) * (2 * RCH) + (i0 & 1);
            const C2* const rrow = rsel + (i0 >> 2) * 2;                     // row q: sample i0 + q TPF
            auto r_at = [&](int i) -> C2 { return rsel[(i >> 2) * 2]; };     // i = i0 (mod 4)
            const T* wr = wrx + hh;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                if (q >= 1 && q <= 13) {
                    // tail_rx/2, shift <= TPF: rows 1..13 neither wrap nor touch the overlap-add margins (nor the window tails)
                    const int n = t + q * TPF + prm.shift;
                    const C2 y = caxpy(g, nz[q], rrow[q * (TPF / 2)]);
                    v[q] = flat_rx ? y : cscale(wr[n], y);
                    continue;
                }
                const int a0 = (q * TPF + prm.shift) & (N - 1);
                const int n = (t + q * TPF + prm.shift) & (N - 1);
                C2 o = cscale(wr[n], caxpy(g, nz[q], r_at(ib + n)));
                if (hh > 0) {
                    const bool wraps = a0 + TPF > N;
                    // overlap-add: the window's tail n + N (extra x = n + hh) and its head n - N (extra x = n - (N - hh))
                    if (wraps || a0 < hh) { if (n < hh) o = caxpy(wr[n + N], caxpy(g, (n + hh >= TPF) ? nx[1] : nx[0], r_at(ib + n + N)), o); }
                    if (wraps || a0 + TPF > N - hh) { if (n >= N - hh) o = caxpy(wr[n - N], caxpy(g, nx[0], r_at(ib + n - N)), o); }
                }
                v[q] = o;
            }
            fft_regs<T, N, -1, FPP>(v, t, xb, tw, slot);
            const uint4 wv = symw[se * TPF + t];
            const uint32_t w[4] = {wv.x, wv.y, wv.z, wv.w};
            // pilot (wofdm_simulation.py:223): the pilot's threads publish Y0, then every thread turns one bin into the
            // equaliser tap G[k] = X0[k] / Y0[k] (lattice units)
            TCV2_STAMP(9);
            if (rank == 0) {
                if (se == 0) {
#pragma unroll
                    for (int q = 0; q < 16; ++q) geq[t + q * TPF] = v[q];
                }
                __syncthreads();
                TCV2_STAMP(10);
                const unsigned char* pil = reinterpret_cast<const unsigned char*>(symw);
                for (int k = tid; k < N; k += NT) {
                    const C2 y0 = geq[k];
                    const C2 x0 = qlut[pil[(k % TPF) * 16 + k / TPF]];
                    C2 gk = cscale(((TCV2_FOLD_SLICER && !VERIFY) ? (T)0.5 : (T)1) * recip(y0.x * y0.x + y0.y * y0.y), cmulc(x0, y0));
                    if (!HS && prm.guard > 0 && !bin_active<N>(k, prm.guard)) gk = mk2<T>(0, 0);
                    geq[k] = gk;
                    if constexpr (CL > 1) {
#pragma unroll
                        for (int r = 1; r < CL; ++r) cooperative_groups::this_cluster().map_shared_rank(geq, r)[k] = gk;
                    }
                }
            }
            if (nvar > 1) build_qtx(var + 1 < nvar ? var + 1 : 0);   // (the Tx stage's table of the next window pair)
            frame_sync<CL>();
            if (act && sb + s > 0) {
                // decisions of four sub-carriers packed like the sent level codes (byte q & 3 of word q >> 2): one XOR per
                // word, the bit errors through the Gray map of the XOR, the symbol errors as its non-zero bytes
#pragma unroll
                for (int gq = 0; gq < 4; ++gq) {
                    uint32_t d4 = 0;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int q = 4 * gq + b, k = t + q * TPF;
                        uint32_t dq;
                        C2 e;
                        if constexpr (TCV2_FOLD_SLICER && !VERIFY) {
                            const C2 gh = geq[k];                                          // G[k] / 2
                            const T off = (T)0.5 * (T)(m - 2), top = (T)(m - 1);
                            const C2 y = fma2(rotj(v[q]), mk2<T>(gh.y, gh.y), fma2(v[q], mk2<T>(gh.x, gh.x), mk2<T>(off, off)));   // :231, :233
                            dq = (__float2uint_ru(fminf(y.x, top)) << hb) | __float2uint_ru(fminf(y.y, top));
                            e = y;
                        } else {
                            e = cmul(v[q], geq[k]);                                        // :231
                            dq = (uint32_t)slice_index(e, hb);                             // :233
                        }
                        d4 |= dq << (8 * b);
                        if constexpr (VERIFY) {
                            const size_t o = ((size_t)f * (prm.S - 1) + (sb + s - 1)) * N + k;
                            prm.eq_out[o] = make_double2((double)e.x * prm.qscale, (double)e.y * prm.qscale);
                            prm.dec_out[o] = levels_to_idx((int)(dq >> hb), (int)(dq & (m - 1)), hb, m, prm.constellation);
                        }
                    }
                    const uint32_t x = d4 ^ w[gq];
                    bit_cnt += code_bit_errors(x, gxm);                                    // :235 (bits) ...
                    sym_cnt += __popc((((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u);   // ... and symbols: bytes that differ
                    if constexpr (RES) { if (prm.res_bins && x) res_add4(racc + 2 * N * var, x, gxm, t + 4 * gq * TPF, TPF); }
                }
            }
        }
        bit_cnt = warp_sum(bit_cnt);
        sym_cnt = warp_sum(sym_cnt);
#if TCV2_TRACE
        TCV2_STAMP(11);
        if (trace_on) {
            __syncthreads();
            if (tid == 0) {
                const long long t0 = trace_buf[0];
                for (int w = 0; w <= NW; ++w) {
                    printf("TRACE it %d warp %d:", trace_it - 1, w);
                    for (int k = 0; k < 12; ++k) printf(" %lld", trace_buf[w * 12 + k] - t0);
                    printf("\n");
                }
            }
            __syncthreads();
        }
#endif
        if constexpr (RES) {
            if (!prm.res_bins && lane == 0) {            // per-cell totals: the per-warp atomics at the cell's address
                atomicAdd(prm.counters + 2 * (var * ncell + rcell), (unsigned long long)bit_cnt);
                atomicAdd(prm.counters + 2 * (var * ncell + rcell) + 1, (unsigned long long)sym_cnt);
            }
        } else if (lane == 0) {
            if constexpr (VERIFY) {
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.bit_err_f) + f, (unsigned long long)bit_cnt);
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.sym_err_f) + f, (unsigned long long)sym_cnt);
            } else {
                atomicAdd(prm.counters + 2 * (var * prm.n_snr + si), (unsigned long long)bit_cnt);
                atomicAdd(prm.counters + 2 * (var * prm.n_snr + si) + 1, (unsigned long long)sym_cnt);
            }
        }
        // No barrier here: what the next frame's prologue and Tx stage overwrite (the split stream over r, the symbol words,
        // the taps operand, the exchange regions over the parked noise) was last read before the pilot barriers above by
        // every thread; geq, red and the tensor-memory accumulators are rewritten only behind the next frame's own barriers.
        if (TCV2_DEBUG_BARRIERS) frame_sync<CL>();
      }   // window pairs
        f += df;
        if constexpr (!VERIFY) {
            fe += de;
            if (fe >= prm.ensemble) { fe -= prm.ensemble; ++ci; }
            ci += dc;
            if (ci >= prm.C) { ci -= prm.C; ++si; }
            si += ds;
        }
        if constexpr (RES) {
            if (prm.seg) { g += df; seg_frame(prm, g, f, si, ci); }   // (replaces the incremental decode)
            if (prm.res_bins) {                          // uniform: the next frame's cell, the frame count, the last frame
                const int nc = prm.res_chan ? si * prm.C + ci : si;
                if (nc != rcell || ++rfr >= rlim || j + nslots >= prm.n_frames) {
                    // the working warps only (the MMA warp keeps its own barrier sequence): every decision of the cell is added
                    asm volatile("bar.sync %0, %1;" :: "n"(TCV2_BAR_RES), "n"(NT) : "memory");
                    res_flush(racc, nvar * N, N, ncell * N, prm.counters + (size_t)rcell * N * 2, tid, NT);
                    rcell = nc; rfr = 0;
                }
            } else {
                rcell = prm.res_chan ? si * prm.C + ci : si;
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    frame_sync<CL>();                              // (nobody leaves while a peer may still read its shared memory)
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(TMEM_COLS) : "memory");
}

}  // namespace wofdm
