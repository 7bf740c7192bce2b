// mask_kernel.cuh -- Tx side of the channel-mask BER variant (SURVEY.md section 8f-1, matlab/main_channel_mask.m).
//
// One CTA builds the serialised, MASKED Tx stream of one frame and writes it to HBM for K1 (BerParams::tx_stream):
// the same Philox symbol draws as K1 (so Rx can redraw them), guard band, register IFFT, CP/CS + Tx window, then the
// DFT-domain raised-cosine mask of gen_tx_ofdm / dft_rc_filt (main_channel_mask.m:384-417): per symbol the zero-padded
// windowed symbol is circularly convolved (mod M = 2 n_tx - 1, not a power of two) with g = IDFT_M(ifftshift(windowRC));
// samples 0..n_tx-1 stay in the symbol, the other n_tx - 1 are added to the start of the NEXT symbol; finally the symbols
// are overlap-added with the frame stride (tx2rx, :420-431).
// The circular convolution of an n_tx-sample symbol equals a LINEAR convolution with the periodic extension of g on
// [-(n_tx-1), M-1], so it runs as forward FFT_P -> multiply by the precomputed response Gp -> inverse FFT_P with
// P = 8N >= 4 n_tx - 3 (register FFTs of fft_regs.cuh, P/16 threads per transform).  fp32.
#pragma once
#include <type_traits>
#include "ber_kernel.cuh"

namespace wofdm {

struct MaskParams {
    int N, cp, cs, tail_tx, bits, S, n_tx, stride, constellation, guard;
    int M;                         // 2 n_tx - 1
    const float* win_tx;           // [n_tx], v_tx * qam_scale / N (the K1 table)
    const float2* tw;              // twiddles of the N-point FFT (the K1 table)
    const float2* twp;             // twiddles of the P-point FFT
    const float2* Gp;              // [P] FFT_P of the periodic extension of the mask's impulse response, times 1/P
    unsigned long long seed;
    long long frame_begin, frame_step, n_frames;
    float2* stream;                // [n_frames][tail_tx + S*stride]
};
// SEG instantiations (frame segments): frame_begin + j*frame_step is a local index into the segment table seg[n_seg][4],
// decoded by seg_frame (BerParams::seg) with C channels and `ensemble` ensemble indices per point.  (A struct of its own:
// MaskParams keeps its size, and with it the code of the unsegmented kernel.)
struct MaskSegParams : MaskParams {
    const long long* seg;
    int n_seg, C;
    long long ensemble;
};

template <int N> struct MaskSmem {
    using PN = FftPlan<N>;
    static constexpr int P = 8 * N;                        // linear-convolution length: >= 4 n_tx - 3 for n_tx <= 2N
    using PP = FftPlan<P>;
    static constexpr int NT = 256, FPP = NT / PN::TPF, FPP_P = NT / PP::TPF;
    static_assert(FPP_P >= 1, "the big transform must fit one CTA");
    static constexpr int XCH = (FPP * PN::XLEN > FPP_P * PP::XLEN) ? FPP * PN::XLEN : FPP_P * PP::XLEN;   // shared exchange
    static size_t bytes(int S, int stride, int tail_tx) {
        const size_t body = (size_t)tail_tx + (size_t)S * stride;
        return ((size_t)S * N + XCH + PN::NTW + PP::NTW + 256 + body + 8) * sizeof(float2);
    }
};

template <int N, bool SEG = false>
__global__ void __launch_bounds__(256) tx_mask_kernel(const std::conditional_t<SEG, MaskSegParams, MaskParams> p) {
    using MS = MaskSmem<N>;
    using PN = typename MS::PN;
    using PP = typename MS::PP;
    constexpr int NT = 256, TPF = PN::TPF, FPP = MS::FPP, P = MS::P, TPFP = PP::TPF, FPPP = MS::FPP_P;
    extern __shared__ __align__(16) unsigned char msm[];
    const int tid = threadIdx.x, slot = tid / TPF, t = tid % TPF;
    const int slotp = tid / TPFP, tp = tid % TPFP;
    const int S = p.S, n_tx = p.n_tx, stride = p.stride, M = p.M;
    const int body = p.tail_tx + S * stride;
    const int hb = p.bits >> 1, m = 1 << hb;
    float2* xs = reinterpret_cast<float2*>(msm);           // [S][N] un-windowed IFFT outputs
    float2* xb = xs + (size_t)S * N;                       // FFT exchange (small and big transforms in turn)
    float2* tw = xb + MS::XCH;
    float2* twp = tw + PN::NTW;
    float2* qlut = twp + PP::NTW;
    float2* us = qlut + 256;                               // [body] the frame stream being accumulated
    for (int i = tid; i < PN::NTW; i += NT) tw[i] = p.tw[i];
    for (int i = tid; i < PP::NTW; i += NT) twp[i] = p.twp[i];
    for (int i = tid; i < 256; i += NT) {
        float2 v = make_float2(0.f, 0.f);
        if (i < (1 << p.bits))                             // level code -> lattice point (ber_kernel.cuh: load_sym_idx)
            v = make_float2((float)(2 * (i >> hb) - (m - 1)), (float)(2 * (i & (m - 1)) - (m - 1)));
        qlut[i] = v;
    }
    __syncthreads();
    BerParams draw = {};                                   // only what load_sym_idx reads
    draw.seed = p.seed; philox_round_keys(p.seed, draw.rk); draw.bits = p.bits; draw.S = S;
    if constexpr (SEG) { draw.C = p.C; draw.ensemble = p.ensemble; draw.seg = p.seg; draw.n_seg = p.n_seg; }
    // symbols per big-transform slot: slot g takes g*half + pass.  At least two, so that symbols filtered at the same time are
    // never neighbours (their stream segments overlap by the Tx tail; S <= FPPP used to put neighbours side by side -- found by
    // the comparison with the mask product, tests/test_drivers_gpu.py::test_channel_mask_product_against_fft_kernel)
    const int half = max(2, (S + FPPP - 1) / FPPP);
    for (long long j = blockIdx.x; j < p.n_frames; j += gridDim.x) {
        long long f = p.frame_begin + j * p.frame_step;
        if constexpr (SEG) { int si, ci; seg_frame(draw, f, f, si, ci); }   // local index -> frame id
        for (int i = tid; i < body; i += NT) us[i] = make_float2(0.f, 0.f);
        // ---- symbols -> IFFT (un-windowed, un-scaled), FPP symbols per pass
        for (int s0 = 0; s0 < S; s0 += FPP) {
            const int s = s0 + slot, se = s < S ? s : S - 1;
            uint32_t w[4];
            load_sym_idx<N, false>(draw, f, se, t, w);
            float2 v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q)
                v[q] = bin_active<N>(t + q * TPF, p.guard) ? qlut[sym_byte(w, q)] : make_float2(0.f, 0.f);
            fft_regs<float, N, +1, FPP>(v, t, xb + slot * PN::XLEN, tw, slot);
#pragma unroll
            for (int q = 0; q < 16; ++q) xs[(size_t)se * N + t + q * TPF] = v[q];
            __syncthreads();
        }
        // ---- mask: slot g filters symbols g*half + pass, pass = 0..half-1.  Concurrent symbols are >= half >= 2 apart
        // (or alone), so the stream segments they add to -- [s*stride, (s+1)*stride + n_tx - 1) -- do not meet.
        for (int pass = 0; pass < half; ++pass) {
            const int s = slotp * half + pass;
            const bool live = s < S;
            const float2* x = xs + (size_t)(live ? s : 0) * N;
            float2 v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int n = tp + q * TPFP;
                v[q] = n < n_tx ? cscale(p.win_tx[n], x[(n - p.cp) & (N - 1)]) : make_float2(0.f, 0.f);
            }
            fft_regs<float, P, -1, FPPP>(v, tp, xb + slotp * PP::XLEN, twp, slotp);
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = cmul(v[q], p.Gp[tp + q * TPFP]);
            fft_regs<float, P, +1, FPPP>(v, tp, xb + slotp * PP::XLEN, twp, slotp);
            // samples 0..n_tx-1 stay in symbol s (stream positions s*stride + n) ...
            if (live) {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int n = tp + q * TPFP;
                    if (n < n_tx) us[s * stride + n] = cadd(us[s * stride + n], v[q]);
                }
            }
            __syncthreads();
            // ... the filter's tail goes to the start of symbol s+1; the last symbol's tail is dropped (:413-416)
            if (live && s + 1 < S) {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int n = tp + q * TPFP;
                    if (n >= n_tx && n < M) us[(s + 1) * stride + (n - n_tx)] = cadd(us[(s + 1) * stride + (n - n_tx)], v[q]);
                }
            }
            __syncthreads();
        }
        float2* dst = p.stream + (size_t)j * body;
        for (int i = tid; i < body; i += NT) dst[i] = us[i];
        __syncthreads();
    }
}

}  // namespace wofdm
