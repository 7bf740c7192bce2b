// ber_kernel.cuh -- K1, the fused Monte-Carlo BER/SER frame kernel (sm_100a).
//
// One CTA processes one frame at a time (S OFDM symbols, symbol 0 = pilot) entirely in shared
// memory and registers, then moves on to its next frame (persistent grid).  Replaces the loop
// body of wOFDMSystem.__run_sim_mc / __run_sim_cp_mc (python/ofdm_utils/wofdm_simulation.py:171-240,
// 328-364) and run_simulation (matlab/main_BER_calculation.m:245-273), in the structured form of
// SURVEY.md App. A.2 instead of the reference's dense tx_mat / rx_mat products:
//
//   draws (Philox or injected) -> QAM map -> IFFT -> CP/CS + Tx window -> overlap-add of the Tx
//   tails into the frame stream -> L-tap channel convolution -> exact-SNR AWGN (frame-wide power
//   sums) -> Rx window -> overlap-add -> circular shift -> FFT -> pilot one-tap equaliser ->
//   hard slicing -> XOR/popcount error counters (warp shuffles, one atomic per warp).
//
// Two policies share this source:
//   TC == 0  "staged": any L, any tail sizes; convolution output staged in a second buffer, noise
//            regenerated in the second pass.  Used for fp64 and for shapes without a tuned variant.
//   TC  > 0  "regs"  : each thread owns one chunk of <= TC consecutive stream samples; the chunk's
//            convolution output stays in registers across the frame-wide power reduction (its noise,
//            generated inside the same loop, is parked in shared memory), all LB taps live in
//            registers.  fp32 production path.
// CIRC (regs policy, CL == 1): the ISI-free interior of every symbol -- outputs whose L inputs all lie in the flat part
// of that symbol's own Tx window, stride - (tail_tx + L - 1) of stride samples -- is a CIRCULAR convolution of the
// symbol with the taps, so it is taken as IFFT(H o X) (one more register FFT per symbol) instead of L complex MACs
// per sample; only the first tail_tx + L - 1 outputs of every symbol (previous tail, prefix, window head) keep the
// direct form.  Same results up to rounding; the host checks that the window really is flat there.
// CL > 1 (regs policy): a thread-block cluster of CL CTAs shares one frame, S/CL consecutive OFDM symbols and
// their part of the frame stream per CTA (N = 1024: the stream plus the parked noise is 278 KB, more than one SM
// holds).  The CTAs meet three times per frame through distributed shared memory: the Tx tail and the L-1
// convolution halo of the previous CTA's last symbol, the frame-wide power sums, and the pilot's equaliser taps.
// VERIFY = true replaces the Philox draws by caller-injected symbols/noise/channel per frame and
// writes the equalised symbols and decisions back (same arithmetic, same code).
#pragma once
#include <cooperative_groups.h>
#include "common.cuh"
#include "fft_regs.cuh"

namespace wofdm {

struct BerParams {
    // system (SURVEY.md App. A.1)
    int N, cp, cs, tail_tx, tail_rx, rm, shift, bits, S;
    int n_tx, stride, L;
    int noise_norm, constellation;
    int flat_tx, flat_rx;      // tensor-core kernel (ber_tconv2.cuh): the window is one value between its tails (and cp, cs >= tail_tx
                               // for Tx): that value moves into the constellation table / is divided out, the flat rows skip the product
                               // (bit v = window pair v of a multi-variant plan)
    int nvar;                  // ber_tconv2.cuh: window pairs evaluated on every frame's symbols in one launch (<= 1: one);
                               // win_tx / win_rx hold nvar tables back to back, counters are [nvar][n_snr][2]
    int guard;                 // null sub-carriers on each side of the centred spectrum (main_channel_mask.m:55,388-391)
    const float2* tx_stream;   // staged policy and TXS instantiations: the serialised Tx stream of local frame j at [j][tail_tx + S*stride],
                               // produced by tx_mask_kernel (channel-mask variant); the Tx stage then only redraws the indices
    int chunk;                 // B: noise block = samples of the frame stream owned by one thread (regs policy);
                               // stream sample i uses draw (i/B)*(B+1) + i%B (B odd: blocks start on a Philox pair);
                               // 0: stream sample i uses draw i (tensor-core convolution policy, ber_tconv.cuh)
    int use_global;            // staged policy: frame buffers live in global scratch
    int split, split_nt;       // CL > 1: stream samples per CTA and threads per CTA (noise block g = rank*NT + local/B); else 0
    int n48;                   // 1: 48-bit noise draws in receiver layout (ber_tconv2.cuh): noise_draw48
    // device tables, element type T / V2<T>
    const void* win_tx;        // [n_tx]   v_tx * qam_scale / N
    const void* win_rx;        // [N + tail_rx]
    const void* tw;            // FFT twiddle sections
    const void* chan;          // V2<T>[C][L]      (verify: [F][L])
    const void* snr_lin;       // T[n_snr] = 10^(-snr/10)   (verify: [F])
    int C, n_snr;
    long long ensemble;
    // production
    unsigned long long seed;
    uint32_t rk[20];           // Philox round keys of `seed` (philox_round_keys; set together with seed)
    unsigned variant;
    long long frame_begin, frame_step, n_frames;   // frame ids f = frame_begin + j*frame_step, j < n_frames
    unsigned long long* counters;                  // [n_snr][2] = {bit_err, sym_err}
    // verify
    const int32_t* sym_idx;    // [F][S][N]
    const double2* noise_in;   // [F][noise_len]
    double2* eq_out;           // [F][S-1][N]
    int32_t* dec_out;          // [F][S-1][N]
    long long* bit_err_f;      // [F]
    long long* sym_err_f;      // [F]
    long long noise_len;
    double qscale;             // constellation amplitude factor (eq_out is reported in signal units)
    // staged policy with use_global: 2 * scratch_elems V2<T> per CTA
    void* scratch;
    long long scratch_elems;
    // TXY instantiations of ber_tconv2.cuh (channel-mask chain): instead of tx_stream, the mask product's output (mask_gemm.cu),
    // one column of tx_yp floats per symbol (local frame j, symbol s: column j*S + s); the loader does the overlap-adds itself
    const float* tx_y;
    int tx_yp;
    // RES instantiations (wofdm_ber_run_resolved): counters are [nvar][cell][bins][2] with cell = si*C + ci (res_chan) or si,
    // bins = N (res_bins: one pair per sub-carrier, accumulated in shared memory) or 1 (the per-warp atomics, re-addressed)
    int res_chan, res_bins;
    // RES instantiations, frame segments (wofdm_ber_run_segments / _adaptive): seg != nullptr makes frame_begin + j*frame_step
    // a LOCAL index g into the segment list, seg[k] = {g0, snr_idx, e_begin, e_count} (g0: local index of its first frame,
    // ascending), channel-major inside a segment; the frame id is f = (snr_idx*C + c)*ensemble + e_begin + e (seg_frame)
    const long long* seg;
    int n_seg;
    // TXY instantiations with nvar > 1 (wofdm_ber_run_masked_multi): window pair v reads its columns at tx_y + v * tx_ypair
    long long tx_ypair;
};

// ---- constellation helpers (oracle/wofdm_oracle.py: idx_to_levels / levels_to_idx) --------------
__device__ __forceinline__ int gray_dec4(int g) { g ^= g >> 1; g ^= g >> 2; return g; }
__device__ __forceinline__ int gray_enc(int v) { return v ^ (v >> 1); }

__device__ __forceinline__ void idx_to_levels(int idx, int hb, int m, int conv, int& a, int& c) {
    if (conv == 0) { a = idx >> hb; c = idx & (m - 1); }
    else { a = gray_dec4(idx >> hb); c = (m - 1) - gray_dec4(idx & (m - 1)); }
}
__device__ __forceinline__ int levels_to_idx(int a, int c, int hb, int m, int conv) {
    return conv == 0 ? ((a << hb) | c) : ((gray_enc(a) << hb) | gray_enc((m - 1) - c));
}
// nearest level on the odd-integer lattice, ties towards the lower level (first minimum of the
// reference's argmin, wofdm_simulation.py:163): ceil(v/2 + (m-2)/2), clamped to [0, m-1]
// (the float -> unsigned conversion saturates at 0, which is the lower clamp)
__device__ __forceinline__ int slice_level(float v, int m) {
    const unsigned lv = __float2uint_ru(fmaf(v, 0.5f, 0.5f * (float)(m - 2)));
    return (int)min(lv, (unsigned)(m - 1));
}
__device__ __forceinline__ int slice_level(double v, int m) {
    const unsigned lv = __double2uint_ru(fma(v, 0.5, 0.5 * (double)(m - 2)));
    return (int)min(lv, (unsigned)(m - 1));
}
// (re level << hb) | (im level), m = 1 << hb levels per axis; float: one packed FMA for both axes
__device__ __forceinline__ int slice_index(float2 e, int hb) {
    const int m = 1 << hb;
    const float off = 0.5f * (float)(m - 2);
    const float2 y = fma2(e, make_float2(0.5f, 0.5f), make_float2(off, off));
    const unsigned la = min(__float2uint_ru(y.x), (unsigned)(m - 1)), lc = min(__float2uint_ru(y.y), (unsigned)(m - 1));
    return (int)((la << hb) | lc);
}
__device__ __forceinline__ int slice_index(double2 e, int hb) {
    const int m = 1 << hb;
    return (slice_level(e.x, m) << hb) | slice_level(e.y, m);
}

// Guard band (matlab/main_channel_mask.m:388-391: zeros on both sides of the centred spectrum, ifftshift): FFT bin k
// carries data iff guard <= (k + N/2) mod N < N - guard.  A null bin takes constellation byte 255 on the Tx side
// (qlut[255] = 0: nothing is sent there and the pilot's equaliser tap X0/Y0 is forced to 0) and the slicer's own
// decision for 0 + 0i as its stored index, so it can never count as an error.
template <int N> __device__ __forceinline__ bool bin_active(int k, int guard) {
    const int c = (k + N / 2) & (N - 1);
    return c >= guard && c < N - guard;
}

// Symbols travel through the kernels as LEVEL CODES, one byte per sub-carrier: (re level << hb) | im level, levels
// 0..m-1 <-> lattice points 2*level - (m-1).  A production draw IS a level code (uniform over the alphabet either way);
// the constellation index of the convention (python natural order / MATLAB Gray) is levels_to_idx(code) and only exists
// at the boundary: verify mode converts the injected indices on load and the decisions on store, wofdm_ber_draws exports
// indices.  In code space the slicer's output needs no table, a symbol error is a non-zero byte of (decided ^ sent), and
// the bit errors are popc(x ^ ((x >> 1) & gray_mask)): both conventions' bit maps are GF(2)-linear in the level bits
// (natural: identity; Gray per axis: v ^ (v >> 1), and MATLAB's inverted imaginary axis m-1-c = c ^ (m-1) cancels in the XOR).
__host__ __device__ __forceinline__ uint32_t gray_xor_mask(int bits, int constellation) {
    const int hb = bits >> 1;
    if (constellation == 0 || hb < 2) return 0u;
    const uint32_t fm = (1u << (hb - 1)) - 1u;           // v >> 1 stays inside its own field
    return (fm | (fm << hb)) * 0x01010101u;
}
// bit errors of four packed level codes (x = decided ^ sent)
__device__ __forceinline__ unsigned code_bit_errors(uint32_t x, uint32_t gmask) { return __popc(x ^ ((x >> 1) & gmask)); }

// 16 level codes (one byte each) of OFDM symbol s for thread t: sub-carriers t + q*TPF
// (BITS > 0: the bits per sub-carrier of a kernel compiled for one geometry, else prm.bits)
template <int N, bool VERIFY, int BITS = 0>
__device__ __forceinline__ void load_sym_idx(const BerParams& prm, long long f, int s, int t, uint32_t (&w)[4]) {
    constexpr int TPF = N / 16;
    if constexpr (VERIFY) {
        const int32_t* src = prm.sym_idx + ((size_t)f * prm.S + s) * N;
        const int hb = prm.bits >> 1, m = 1 << hb;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t x = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                int a, c;
                idx_to_levels(src[t + (4 * j + b) * TPF] & 0xff, hb, m, prm.constellation, a, c);
                x |= (uint32_t)((a << hb) | c) << (8 * b);
            }
            w[j] = x;
        }
    } else {
        const uint4 r = philox4x32_10_rk(make_uint4((uint32_t)f, (uint32_t)((unsigned long long)f >> 32),
                                                    (uint32_t)(s * TPF + t), STREAM_SYM), prm.rk);
        const uint32_t mask = ((1u << (BITS > 0 ? BITS : prm.bits)) - 1u) * 0x01010101u;
        w[0] = r.x & mask; w[1] = r.y & mask; w[2] = r.z & mask; w[3] = r.w & mask;
    }
}
// (one PRMT: byte q&3 of the word, zero-extended)
__device__ __forceinline__ int sym_byte(const uint32_t (&w)[4], int q) { return (int)__byte_perm(w[q >> 2], 0u, 0x4440u + (unsigned)(q & 3)); }

// complex noise draws 2q and 2q+1 of frame f
template <typename T>
__device__ __forceinline__ void noise_pair(const BerParams& prm, long long f, uint32_t q, V2<T>& n0, V2<T>& n1) {
    const uint4 r = philox4x32_10_rk(make_uint4((uint32_t)f, (uint32_t)((unsigned long long)f >> 32), q,
                                                STREAM_NOISE + prm.variant), prm.rk);
    gauss_quad(r, n0, n1, T());
}
// ---- 48-bit noise draws in receiver layout (ber_tconv2.cuh) --------------------------------------------------------
// The tensor-core kernels draw the noise of a frame where the receiver uses it: thread t (of N/16 = TPF) of symbol s's
// transform holds, in registers, the noise of the 16 samples its FFT rows gather -- block offsets n = (t + q TPF + shift)
// mod N, q = 0..15, stream position s stride + rm + hh + n -- plus its share of the symbol's other stride - N samples,
// the "extras" x = 0 .. XA-1 laid along the ring of threads (thread (base + x) mod TPF, level x / TPF):
//   x < hh            head of the Rx window's overlap-add, block index k = x          (added to n = N - hh + x)
//   hh <= x < 2 hh    its tail,                            k = N + x                  (added to n = x - hh)
//   2 hh <= x < XA    the rm samples in front of the block that the receiver drops (they count in the noise power only)
//   x >= XA           last symbol, noise_norm = 1: the tail_tx + L - 1 samples behind the frame (full-convolution sums)
// base = (N - hh - shift) mod TPF puts every overlap-add sample into the thread that needs it.
// 48 random bits per complex sample: a 32-bit radius word and a 16-bit angle (65 536 phases).  Philox calls of (s, t):
// counter index ((s TPF + t) N48_CALLS + c); c = 3 g + {0, 1, 2} serve the main samples q = 8 g + e: radius = word e of
// (call 3g, call 3g+1), angle = half e & 1 of word e >> 1 of call 3g+2; c = 6, 7, ... give the words V[0..) of the extras:
// levels 2 j, 2 j + 1 take their angles from the halves of V[3 j] and their radii from V[3 j + 1], V[3 j + 2].
constexpr int N48_MAXLEV = 16;                                   // extra levels a symbol may have (pairs of two)
constexpr int N48_MAXLEV_SHORT = 6;                             // ... in the kernels for L <= 21 (inline draws)
constexpr int N48_CALLS = 6 + (3 * (N48_MAXLEV / 2) + 3) / 4;     // Philox calls reserved per (symbol, thread): 12
// (var: window pair of a multi-variant launch; its noise stream is that of a single launch with variant + var)
__device__ __forceinline__ uint4 noise48_call(const BerParams& prm, long long f, uint32_t q, int var = 0) {
    return philox4x32_10_rk(make_uint4((uint32_t)f, (uint32_t)((unsigned long long)f >> 32), q, STREAM_NOISE + prm.variant + (uint32_t)var), prm.rk);
}
// two complex samples: radius words u0, u1, angles = low / high half of aw.  Same arithmetic as gauss_quad.
__device__ __forceinline__ void gauss_quad48(uint32_t u0, uint32_t u1, uint32_t aw, float2& n0, float2& n1) {
    const float2 u = fma2(make_float2(__uint2float_rn(u0), __uint2float_rn(u1)),
                          make_float2(2.3283064365386963e-10f, 2.3283064365386963e-10f),
                          make_float2(1.1641532182693481e-10f, 1.1641532182693481e-10f));
    float2 lg, rr;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg.x) : "f"(u.x));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg.y) : "f"(u.y));
    const float2 t = mul2(lg, make_float2(-1.3862943611198906f, -1.3862943611198906f));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rr.x) : "f"(t.x));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rr.y) : "f"(t.y));
    // theta = 2 pi a / 65536, a the signed 16-bit half: in [-pi, pi)
    const float2 th = mul2(make_float2(__int2float_rn((int32_t)(aw << 16)), __int2float_rn((int32_t)(aw & 0xffff0000u))),
                           make_float2(1.4629180792671596e-09f, 1.4629180792671596e-09f));
    float s0, c0, s1, c1;
    asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s0) : "f"(th.x));
    asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c0) : "f"(th.x));
    asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s1) : "f"(th.y));
    asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c1) : "f"(th.y));
    n0 = mul2(make_float2(c0, s0), make_float2(rr.x, rr.x));
    n1 = mul2(make_float2(c1, s1), make_float2(rr.y, rr.y));
}
__device__ __forceinline__ uint32_t u4_word(const uint4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
// geometry of the extras of a frame (host and device)
struct N48Geom { int tpf, hh, xa, tailx, base; };
__host__ __device__ __forceinline__ N48Geom n48_geom(const BerParams& prm) {
    N48Geom g;
    g.tpf = prm.N / 16; g.hh = prm.tail_rx >> 1; g.xa = prm.stride - prm.N;
    g.tailx = prm.noise_norm == 1 ? prm.tail_tx + prm.L - 1 : 0;
    g.base = (prm.N - g.hh - prm.shift) & (g.tpf - 1);
    return g;
}
// frame offset (relative to the symbol's first stream sample) of extra x
__host__ __device__ __forceinline__ int n48_extra_offset(const BerParams& prm, const N48Geom& g, int x) {
    return x < g.hh ? prm.rm + x : x < 2 * g.hh ? prm.rm + prm.N + x : x < g.xa ? x - 2 * g.hh : prm.stride + (x - g.xa);
}
// noise of stream sample p (export path, wofdm_ber_draws / noise_at)
__device__ __forceinline__ float2 noise_draw48(const BerParams& prm, long long f, int p) {
    const N48Geom g = n48_geom(prm);
    const int s = min(p / prm.stride, prm.S - 1), o = p - s * prm.stride;
    int t, wr, wa, half, cr, ca;            // thread; radius word / angle word (call, index)
    if (o >= prm.rm + g.hh && o < prm.rm + g.hh + prm.N) {
        const int tp = (o - prm.rm - g.hh - prm.shift) & (prm.N - 1);
        t = tp & (g.tpf - 1);
        const int q = tp / g.tpf, gq = q >> 3, e = q & 7;
        cr = 3 * gq + (e >> 2); wr = e & 3; ca = 3 * gq + 2; wa = e >> 1; half = e & 1;
    } else {
        const int x = o < prm.rm ? 2 * g.hh + o : o < prm.rm + g.hh ? o - prm.rm : o < prm.stride ? o - prm.rm - prm.N : g.xa + o - prm.stride;
        t = (g.base + x) & (g.tpf - 1);
        const int lev = x / g.tpf, j = lev >> 1;
        const int ia = 3 * j, ir = 3 * j + 1 + (lev & 1);
        cr = 6 + (ir >> 2); wr = ir & 3; ca = 6 + (ia >> 2); wa = ia & 3; half = lev & 1;
    }
    const uint32_t q0 = (uint32_t)(s * g.tpf + t) * (uint32_t)N48_CALLS;
    const uint32_t uw = u4_word(noise48_call(prm, f, q0 + (uint32_t)cr), wr), aw = u4_word(noise48_call(prm, f, q0 + (uint32_t)ca), wa);
    float2 n0, n1;
    gauss_quad48(uw, uw, aw, n0, n1);
    return half ? n1 : n0;
}

// noise of stream sample i (any policy): draw index (i/B)*(B+1) + i%B
template <typename T>
__device__ __forceinline__ V2<T> noise_at(const BerParams& prm, long long f, int i) {
    const int B = prm.chunk;
    if (prm.n48) {             // (fp32 kernels only)
        const float2 z = noise_draw48(prm, f, i);
        return mk2<T>((T)z.x, (T)z.y);
    }
    if (B == 0) {              // draw = position
        V2<T> n0, n1;
        noise_pair<T>(prm, f, (uint32_t)(i >> 1), n0, n1);
        return (i & 1) ? n1 : n0;
    }
    int k0 = 0;
    if (prm.split > 0) {       // frame shared by a cluster: blocks are numbered per CTA
        const int r = min(i / prm.split, prm.S * prm.stride / prm.split - 1);
        i -= r * prm.split;
        k0 = r * prm.split_nt;
    }
    const int kl = i / B;
    const int k = k0 + kl;
    const int d = k * (B + 1) + (i - kl * B);
    V2<T> n0, n1;
    noise_pair<T>(prm, f, (uint32_t)(d >> 1), n0, n1);
    return (d & 1) ? n1 : n0;
}

template <typename T> __device__ __forceinline__ V2<T> to_v2(double2 d) { return mk2<T>((T)d.x, (T)d.y); }

// shared-memory carve-up, computed identically on host (for the launch) and device
struct BerSmem {
    int pad;        // zero samples in front of the frame stream (covers every negative tap index)
    int flen;       // frame-stream buffer elements incl. pad and tail slack (0: lives in global scratch)
    int xlen;       // second buffer elements: staged -> conv output / FFT exchange; regs -> noise / FFT exchange
    int off_x, off_tw, off_geq, off_hf, off_taps, off_wtx, off_wrx, off_red, off_qlut, off_dlut, off_gmask, off_symw;   // byte offsets
    int off_lo, off_bt, off_bar;   // tensor-core convolution policy (ber_tconv2.cuh): lo half of the split stream, taps operand, mbarrier
    size_t bytes;
    int off_res;    // RES instantiations: per-sub-carrier error accumulators, uint32 {bit, sym} per (window pair, bin)
};

// Per-sub-carrier error counts of the RES instantiations (wofdm_ber_run_resolved).  A CTA adds the errors of every decided
// symbol into 32-bit shared accumulators racc[var][k] = {bit, sym} and moves them to the u64 counters of its current cell only
// when the cell (SNR point, or SNR point x channel) of its next frame differs, before a 32-bit accumulator could wrap, and at
// its last frame.  Frames f = (si*C + ci)*ensemble + e are taken round-robin, so a CTA stays in one cell for ensemble / (frames
// in flight) frames in a row.  Zero accumulators are skipped; the shared atomics of a frame only touch bins with an error.
// add the errors of x = decided ^ sent (four level codes, byte b = bin k0 + b*kstep) to the accumulators
__device__ __forceinline__ void res_add4(uint32_t* racc, uint32_t x, uint32_t gxm, int k0, int kstep) {
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const uint32_t xb = (x >> (8 * b)) & 0xffu;
        if (xb) {
            uint32_t* a = racc + 2 * (k0 + b * kstep);
            atomicAdd(a, code_bit_errors(xb, gxm));
            atomicAdd(a + 1, 1u);
        }
    }
}
// move the n accumulator pairs of this CTA into dst (pair e -> dst[2 * (e / nb * cstride + e % nb)]) and zero them.
// Ordering, both sides by barriers: callers put one in front (every add of the old cell is done), and the next frame's adds
// come only after the CTA-wide barriers every policy passes before its decisions (the power sums' frame_sync, the pilot's
// barrier), which every thread reaches only after its part of this loop.  A schedule without such a barrier between the
// flush and the next decisions needs a second barrier here.
__device__ __forceinline__ void res_flush(uint32_t* racc, int n, int nb, size_t cstride, unsigned long long* dst, int tid, int nt) {
    for (int e = tid; e < n; e += nt) {
        const unsigned sc = racc[2 * e + 1];
        if (sc == 0u) continue;                        // (no symbol error: no bit error either)
        const unsigned bb = racc[2 * e];
        racc[2 * e] = 0u; racc[2 * e + 1] = 0u;
        unsigned long long* d = dst + 2 * ((size_t)(e / nb) * cstride + (e % nb));
        atomicAdd(d, (unsigned long long)bb);
        atomicAdd(d + 1, (unsigned long long)sc);
    }
}
// local index g of a segment launch -> frame id f, SNR point si, channel ci (BerParams::seg).  Uniform over the CTA (and the
// cluster).  g at or past the end maps to a channel >= C of the last segment: only the loop's exit test follows.
__device__ __forceinline__ void seg_frame(const BerParams& prm, long long g, long long& f, int& si, int& ci) {
    int lo = 0, hi = prm.n_seg - 1;                    // the last segment that starts at or before g
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (prm.seg[4 * mid] <= g) lo = mid; else hi = mid - 1;
    }
    const long long* sg = prm.seg + 4 * lo;
    const long long r = g - sg[0], ec = sg[3], c = r / ec;
    si = (int)sg[1];
    ci = (int)c;
    f = ((long long)si * prm.C + c) * prm.ensemble + sg[2] + (r - c * ec);
}

// frames between flushes such that no 32-bit accumulator wraps: a frame adds at most S * bits bit errors to a bin
__host__ __device__ __forceinline__ unsigned res_frame_limit(int S, int bits) { return 0xffffffffu / (unsigned)(S * (bits > 1 ? bits : 1)); }

template <typename T, int N, int NT, int TC, int LB, bool RES = false>
__host__ __device__ inline BerSmem ber_smem_layout(int S, int stride, int tail_tx, int tail_rx, int L, int chunk,
                                                   int use_global) {
    using P = FftPlan<N>;
    constexpr int FPP = NT / P::TPF;
    constexpr int E = (int)sizeof(V2<T>);
    BerSmem m;
    constexpr int lbs = LB > 0 ? LB : 1;
    const int lpad = TC > 0 ? ((L + lbs - 1) / lbs) * lbs : L;
    m.pad = (lpad + 1) & ~1;
    const int body = tail_tx + S * stride;
    const int exch = FPP * P::XLEN;
    if (TC > 0) {
        const int need = body > NT * chunk ? body : NT * chunk;
        m.flen = m.pad + need + TC + 2;
        m.xlen = exch > NT * chunk + 2 ? exch : NT * chunk + 2;   // noise of the frame; FFT exchange in Tx/Rx
    } else {
        m.flen = use_global ? 0 : m.pad + body + 2;
        const int sec = S * stride;
        m.xlen = use_global ? exch : (exch > sec ? exch : sec);
    }
    m.flen = (m.flen + 1) & ~1;
    m.xlen = (m.xlen + 1) & ~1;
    int o = 0;
    o += m.flen * E;                 m.off_x = o;
    o += m.xlen * E;                 m.off_tw = o;
    o += P::NTW * E;                 m.off_geq = o;
    o += N * E;                      m.off_hf = o;     // channel frequency response x flat window value (CIRC)
    o += (TC > 0 ? N : 0) * E;       m.off_taps = o;
    o += (((L > lpad ? L : lpad) + 1) & ~1) * E;   m.off_wtx = o;   // taps, zero-padded to the register block
    o += ((stride + tail_tx + 3) & ~3) * (int)sizeof(T);   m.off_wrx = o;
    o += ((N + tail_rx + 3) & ~3) * (int)sizeof(T);        m.off_red = o;
    o += 64 * (int)sizeof(T);                              m.off_qlut = o;
    o += 256 * E;                                          m.off_dlut = o;
    o += 256;                                              m.off_gmask = o;
    o += P::TPF * 32;                                      m.off_symw = o;     // guard band: two uint4 per thread of a transform
    o += S * P::TPF * 16;                                  // constellation-index words of every (symbol, thread)
    m.off_res = 0;
    if constexpr (RES) { o = (o + 15) & ~15; m.off_res = o; o += N * 8; }
    m.bytes = ((size_t)o + 15) & ~(size_t)15;
    return m;
}

__device__ __forceinline__ float recip(float x) { return __fdividef(1.0f, x); }
__device__ __forceinline__ double recip(double x) { return 1.0 / x; }

// sum of the NW per-warp partials every thread reads after the frame-wide barrier (fixed order:
// the result does not depend on scheduling); r is 16-byte aligned
template <int NW> __device__ __forceinline__ float block_total(const float* r) {
    float s = 0.0f;
    if constexpr (NW % 4 == 0) {
#pragma unroll
        for (int i = 0; i < NW / 4; ++i) { const float4 v = reinterpret_cast<const float4*>(r)[i]; s += (v.x + v.y) + (v.z + v.w); }
    } else {
#pragma unroll
        for (int i = 0; i < NW; ++i) s += r[i];
    }
    return s;
}
template <int NW> __device__ __forceinline__ double block_total(const double* r) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < NW; ++i) s += r[i];
    return s;
}
// g = sqrt(Pr * 10^(-snr/10) / Pn)   (wofdm_simulation.py:135-138)
__device__ __forceinline__ float noise_gain(float pr, float snr_lin, float pn) {
    float g;
    const float q = __fdividef(pr * snr_lin, pn);
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(g) : "f"(q));
    return g;
}
__device__ __forceinline__ double noise_gain(double pr, double snr_lin, double pn) { return sqrt(pr * snr_lin / pn); }

// one output of the direct-form convolution past the kept samples (MATLAB's full-length noise normalisation): taps are
// zero-padded to LB in shared memory, inputs at and beyond `body` do not exist.  Fully unrolled with two accumulators so
// that the few threads which run it do not serialise 2*LB shared-memory latencies in front of the frame-wide barrier.
template <typename T, int LB>
__device__ __forceinline__ V2<T> tail_output(const V2<T>* taps, const V2<T>* ub, int i, int body) {
    V2<T> a0 = mk2<T>(0, 0), a1 = mk2<T>(0, 0);
#pragma unroll
    for (int l = 0; l < LB; ++l) {
        const V2<T> x = (i - l < body) ? ub[i - l] : mk2<T>(0, 0);
        if (l & 1) cmac(a1, taps[l], x); else cmac(a0, taps[l], x);
    }
    return cadd(a0, a1);
}

// barrier over the CTAs of a frame (release/acquire at cluster scope: remote shared-memory traffic is ordered)
template <int CL> __device__ __forceinline__ void frame_sync() {
    if constexpr (CL > 1) cooperative_groups::this_cluster().sync(); else __syncthreads();
}

// TXS: the Tx stage can take the frame's stream from HBM (BerParams::tx_stream, channel-mask variant).  Always possible in
// the staged policy; the register-resident kernels get it as separate instantiations so that the main path keeps its code.
// RES: error counters resolved by sub-carrier and / or channel (BerParams::res_chan / res_bins); in a cluster every CTA keeps
// and flushes the accumulators of its own symbols.  RES && TXS: the twins of the channel-mask chain's TXS kernels
template <typename T, int N, int NT, int TC, int LB, int MINB, bool FULL, bool VERIFY, int CL = 1, bool CIRC = false, bool TXS = false,
          bool RES = false>
__global__ void __launch_bounds__(NT, MINB)
ber_frame_kernel(const BerParams prm) {
    using P = FftPlan<N>;
    using C2 = V2<T>;
    constexpr int TPF = P::TPF;
    constexpr int FPP = NT / TPF;
    static_assert(NT % TPF == 0 && NT % 32 == 0, "threads per CTA must be a multiple of N/16 and 32");
    constexpr bool REGS = TC > 0;
    static_assert(CL == 1 || REGS, "clusters are a feature of the register-resident policy");
    static_assert(!RES || !VERIFY, "resolved counters: production kernels");
    static_assert(!CIRC || (REGS && CL == 1 && N <= NT), "circular-interior policy: regs, one CTA per frame, one bin per thread");
    // Register row q of a thread = sub-carriers / samples t + q*TPF.  Only the outer rows can reach the cyclic
    // prefix / suffix, the Tx heads and the Rx overlap-add; the tuned variants look at ER of them (the host
    // checks cp, cs, tail_tx <= ER*TPF and tail_rx/2, shift <= TPF), the staged policy at all 16.
    constexpr int ER = REGS ? 2 : 16;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x;
    const int slot = tid / TPF, t = tid % TPF;
    // this CTA's share of the frame: S OFDM symbols starting at symbol sb (the whole frame when CL == 1)
    int rank = 0;
    if constexpr (CL > 1) rank = (int)cooperative_groups::this_cluster().block_rank();
    const int S = prm.S / CL, sb = rank * S;
    const int stride = prm.stride, n_tx = prm.n_tx, beta = prm.tail_tx, L = prm.L;
    const int cp = prm.cp, cs = prm.cs;
    const int hh = prm.tail_rx >> 1;
    const int hb = prm.bits >> 1, m = 1 << hb;
    const int sec = S * stride;                 // samples kept after the channel (this CTA's)
    const int body = beta + sec;                // serialised Tx stream length
    const bool last_rank = rank == CL - 1;

    const BerSmem lay = ber_smem_layout<T, N, NT, TC, LB, RES>(S, stride, beta, prm.tail_rx, L, prm.chunk, prm.use_global);
    C2* fbuf = reinterpret_cast<C2*>(smem_raw);
    C2* xbuf = reinterpret_cast<C2*>(smem_raw + lay.off_x);
    C2* tw = reinterpret_cast<C2*>(smem_raw + lay.off_tw);
    C2* geq = reinterpret_cast<C2*>(smem_raw + lay.off_geq);
    C2* hf = reinterpret_cast<C2*>(smem_raw + lay.off_hf);
    C2* taps = reinterpret_cast<C2*>(smem_raw + lay.off_taps);
    T* wtx = reinterpret_cast<T*>(smem_raw + lay.off_wtx);
    T* wrx = reinterpret_cast<T*>(smem_raw + lay.off_wrx);
    T* red = reinterpret_cast<T*>(smem_raw + lay.off_red);
    C2* qlut = reinterpret_cast<C2*>(smem_raw + lay.off_qlut);          // level code -> lattice point
    uint4* symw = reinterpret_cast<uint4*>(smem_raw + lay.off_symw);     // Tx -> Rx: the frame's constellation indices
    uint4* gmask = reinterpret_cast<uint4*>(smem_raw + lay.off_gmask);   // guard band: [t][0] = 0xff in null bytes, [t][1] = stored index there
    C2* rbuf = xbuf;                            // staged: conv output; regs: the frame's noise (both alias the exchange)
    if (!REGS && prm.use_global) {
        C2* g = reinterpret_cast<C2*>(prm.scratch) + (size_t)blockIdx.x * 2 * prm.scratch_elems;
        fbuf = g;
        rbuf = g + prm.scratch_elems;
    }
    C2* const ub = fbuf + lay.pad;              // ub[i] = stream sample i (CTA-local), ub[-pad..-1] = 0 or the halo
    C2* const xb = xbuf + slot * P::XLEN;
    // distributed shared memory: the previous CTA's stream (tail + halo), CTA 0's equaliser taps, every CTA's sums
    // (pulled: a few dozen samples per frame; the power sums and the equaliser taps are PUSHED into every CTA's
    // copy with remote stores, which do not stall, so all their reads are local)
    const C2* prev_ub = ub;
    if constexpr (CL > 1) {
        if (rank > 0) prev_ub = cooperative_groups::this_cluster().map_shared_rank(ub, rank - 1);
    }
    static_assert(CL * (NT / 32) <= 32, "per-warp partial sums of all CTAs must fit the reduction scratch");

    // ---- one-time tables ----
    for (int i = tid; i < P::NTW; i += NT) tw[i] = reinterpret_cast<const C2*>(prm.tw)[i];
    for (int i = tid; i < n_tx; i += NT) wtx[i] = reinterpret_cast<const T*>(prm.win_tx)[i];
    for (int i = tid; i < N + prm.tail_rx; i += NT) wrx[i] = reinterpret_cast<const T*>(prm.win_rx)[i];
    for (int i = tid; i < lay.pad; i += NT) fbuf[i] = mk2<T>(0, 0);
    for (int i = tid; i < (1 << prm.bits); i += NT)                      // level code -> lattice point
        qlut[i] = mk2<T>((T)(2 * (i >> hb) - (m - 1)), (T)(2 * (i & (m - 1)) - (m - 1)));
    if (tid == 0 && prm.bits < 8) qlut[255] = mk2<T>(0, 0);              // the null sub-carrier
    const uint32_t gxm = gray_xor_mask(prm.bits, prm.constellation);
    uint32_t* const racc = reinterpret_cast<uint32_t*>(smem_raw + lay.off_res);   // RES: [N][2] = {bit, sym}
    if constexpr (RES) { for (int i = tid; i < 2 * N; i += NT) racc[i] = 0u; }
    __syncthreads();
    if (prm.guard > 0) {
        const unsigned d0 = slice_index(mk2<T>(0, 0), hb);                // what the slicer makes of a null bin
        for (int tt = tid; tt < TPF; tt += NT) {
            uint32_t ff[4] = {0, 0, 0, 0}, dd[4] = {0, 0, 0, 0};
            for (int q = 0; q < 16; ++q)
                if (!bin_active<N>(tt + q * TPF, prm.guard)) { ff[q >> 2] |= 0xffu << (8 * (q & 3)); dd[q >> 2] |= d0 << (8 * (q & 3)); }
            gmask[2 * tt] = make_uint4(ff[0], ff[1], ff[2], ff[3]);
            gmask[2 * tt + 1] = make_uint4(dd[0], dd[1], dd[2], dd[3]);
        }
        __syncthreads();
    }

    C2 wk = mk2<T>(1, 0);                       // CIRC: exp(-2 pi i tid / N), the step of bin tid's DFT phasor
    if constexpr (CIRC) { float sn, cs_; sincospif(-2.0f * (float)tid / (float)N, &sn, &cs_); wk = mk2<T>((T)cs_, (T)sn); }

    // frame id f = (si*C + ci)*ensemble + e, advanced without per-frame divisions
    const long long fslot = blockIdx.x / CL, nslots = gridDim.x / CL;   // frames in flight on the grid
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
    // RES with a segment table: f above is the local index g, every frame's (f, si, ci) comes from seg_frame
    [[maybe_unused]] long long g = f;
    if constexpr (RES) { if (prm.seg) seg_frame(prm, g, f, si, ci); }
    // RES: cells of the counters and this CTA's current one
    const size_t ncell = RES ? (size_t)prm.n_snr * (prm.res_chan ? prm.C : 1) : 0;
    int rcell = RES ? (prm.res_chan ? si * prm.C + ci : si) : 0;
    unsigned rfr = 0;
    const unsigned rlim = RES ? res_frame_limit(prm.S, prm.bits) : 0u;
    for (long long j = fslot; j < prm.n_frames; j += nslots) {
        if constexpr (VERIFY) { ci = (int)f; si = (int)f; }
        const T snr_lin = reinterpret_cast<const T*>(prm.snr_lin)[si];
        if (tid < (REGS ? (LB > L ? LB : L) : L))   // regs policy: zero-padded to LB, loaded without predicates
            taps[tid] = tid < L ? reinterpret_cast<const C2*>(prm.chan)[(size_t)ci * L + tid] : mk2<T>(0, 0);
        if constexpr (CIRC) {
            // H'[k] = w_flat * sum_l h[l] exp(-2 pi i k l / N), one bin per thread, phasor by recurrence
            __syncthreads();
            if (tid < N) {
                C2 ph = mk2<T>(1, 0), a = mk2<T>(0, 0);
                for (int l = 0; l < L; ++l) { cmac(a, taps[l], ph); ph = cmul(ph, wk); }
                hf[tid] = cscale(wtx[beta], a);
            }
            __syncthreads();
        }

        // =========================== transmitter ===========================
        C2 cv[16];                              // CIRC: interior of the channel output, c[t + q*TPF] (single Tx pass)
        bool tx_done = false;
        if constexpr (TXS || TC == 0) {
            static_assert(!(TXS && (CIRC || CL > 1)), "tx_stream: direct-form, one CTA per frame");
            if (prm.tx_stream != nullptr) {     // uniform: masked Tx stream from tx_mask_kernel (mask_kernel.cuh)
                for (int e = tid; e < S * TPF; e += NT) {
                    const int tt = e % TPF;
                    uint32_t w[4];
                    load_sym_idx<N, VERIFY>(prm, f, e / TPF, tt, w);
                    if (prm.guard > 0) {
                        const uint4 gf = gmask[2 * tt], gd = gmask[2 * tt + 1];
                        w[0] = (w[0] & ~gf.x) | gd.x; w[1] = (w[1] & ~gf.y) | gd.y;
                        w[2] = (w[2] & ~gf.z) | gd.z; w[3] = (w[3] & ~gf.w) | gd.w;
                    }
                    symw[e] = make_uint4(w[0], w[1], w[2], w[3]);
                }
                const float2* src = prm.tx_stream + (size_t)j * body;
                for (int i = tid; i < body; i += NT) ub[i] = mk2<T>((T)src[i].x, (T)src[i].y);
                tx_done = true;
            }
        }
        for (int s0 = 0; s0 < S && !tx_done; s0 += FPP) {
            const int s = s0 + slot;
            const bool act = s < S;
            const int se = act ? s : S - 1;     // idle slots shadow the last symbol (identical stores)
            const bool first = sb + se == 0;    // the frame's first symbol has no predecessor
            C2 v[16];
            {
                uint32_t w[4], wq[4];             // stored indices (Rx compares against them) / Tx look-up indices
                load_sym_idx<N, VERIFY>(prm, f, sb + se, t, w);
#pragma unroll
                for (int jw = 0; jw < 4; ++jw) wq[jw] = w[jw];
                if (prm.guard > 0) {              // uniform: null bins send nothing and store the slicer's 0+0i decision
                    const uint4 gf = gmask[2 * t], gd = gmask[2 * t + 1];
                    const uint32_t ff[4] = {gf.x, gf.y, gf.z, gf.w}, dd[4] = {gd.x, gd.y, gd.z, gd.w};
#pragma unroll
                    for (int jw = 0; jw < 4; ++jw) { wq[jw] = w[jw] | ff[jw]; w[jw] = (w[jw] & ~ff[jw]) | dd[jw]; }
                }
                symw[se * TPF + t] = make_uint4(w[0], w[1], w[2], w[3]);
                if constexpr (CIRC) {
                    // c = w_flat * (h circ x) = IFFT(H' o X)
#pragma unroll
                    for (int q = 0; q < 16; ++q) cv[q] = cmul(qlut[sym_byte(wq, q)], hf[t + q * TPF]);
                    fft_regs<T, N, +1, FPP>(cv, t, xb, tw, slot);
                }
#pragma unroll
                for (int q = 0; q < 16; ++q) v[q] = qlut[sym_byte(wq, q)];
            }
            fft_regs<T, N, +1, FPP>(v, t, xb, tw, slot);
            // CP/CS insertion + Tx window: sample i of symbol s is wtx[i] * x[(i - cp) mod N]
            // (transmitter.py:13-35, 61-87).  Head samples i < tail_tx overlap the previous
            // symbol's falling tail (wofdm_simulation.py:190-203) and are added after the sync.
            C2* const us = ub + se * stride;
            if (cp >= beta) {
                T wv[16];                                 // window loads ahead of the (possibly aliasing) stores
#pragma unroll
                for (int q = 0; q < 16; ++q) wv[q] = wtx[t + q * TPF + cp];
#pragma unroll
                for (int q = 0; q < 16; ++q) us[t + q * TPF + cp] = cscale(wv[q], v[q]);
            } else {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int i = t + q * TPF + cp;
                    if (q >= ER || i >= beta || first) us[i] = cscale(wtx[i], v[q]);
                }
            }
#pragma unroll
            for (int q = 16 - ER; q < 16; ++q) {
                if (q * TPF + TPF > N - cp) {             // uniform: this register row reaches the prefix
                    const int i = t + q * TPF - (N - cp);
                    if (i >= 0 && (i >= beta || first)) us[i] = cscale(wtx[i], v[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < ER; ++q) {
                if (q * TPF < cs) {                        // uniform: ... the suffix
                    const int i = t + q * TPF + cp + N;
                    if (i < n_tx) us[i] = cscale(wtx[i], v[q]);
                }
            }
            frame_sync<CL>();
            // the falling tail of the previous symbol: same buffer, or the previous CTA's (its slack past `sec`)
            const C2* const tl = (CL > 1 && se == 0) ? prev_ub + sec : us;
            if (beta > 0 && act && !first) {
#pragma unroll
                for (int q = 16 - ER; q < 16; ++q) {
                    if (q * TPF + TPF > N - cp) {
                        const int i = t + q * TPF - (N - cp);
                        if (i >= 0 && i < beta) us[i] = caxpy(wtx[i], v[q], tl[i]);
                    }
                }
                if (cp < beta) {
#pragma unroll
                    for (int q = 0; q < ER; ++q) {
                        const int i = t + q * TPF + cp;
                        if (i < beta) us[i] = caxpy(wtx[i], v[q], tl[i]);
                    }
                }
            }
            if constexpr (CL > 1) {
                // convolution halo: the last `pad` stream samples of the previous CTA (none of them is a head)
                // (CL > 1 requires a single pass, S/CL <= FPP: the previous CTA's last symbol is complete here)
                if (rank > 0 && tid < lay.pad) fbuf[tid] = prev_ub[sec - lay.pad + tid];
            }
        }
        __syncthreads();

        // =========================== channel + AWGN ===========================
        // r = conv(h, u)[0:sec] (wofdm_simulation.py:206-209); y = r + sqrt(Pr*10^(-snr/10)/Pn) n
        // with Pr, Pn summed over the whole frame (:135-138).  noise_norm 1: sums over the full
        // convolution, beta+sec+L-1 samples (main_BER_calculation.m:260-261,289-292).
        C2 pr2 = mk2<T>(0, 0), pn2 = mk2<T>(0, 0);
        if constexpr (CIRC) {
            // ---- noise of this thread's block of B stream samples -> shared memory, |n|^2 partial (numbering as in regs)
            const int B = prm.chunk;
            const int i0 = tid * B;
            const int nvalid = FULL ? TC : min(B, max(sec - i0, 0));
            C2* const nb = rbuf + i0;
            constexpr int NPAIR = (TC + 1) / 2;
            const uint32_t q0 = (uint32_t)tid * (uint32_t)((B + 1) >> 1);
#pragma unroll
            for (int p2 = 0; p2 < NPAIR; ++p2) {
                C2 n0, n1;
                if constexpr (VERIFY) {
                    const double2* nin = prm.noise_in + (size_t)f * prm.noise_len + i0;
                    n0 = (2 * p2 < nvalid) ? to_v2<T>(nin[2 * p2]) : mk2<T>(0, 0);
                    n1 = (2 * p2 + 1 < nvalid) ? to_v2<T>(nin[2 * p2 + 1]) : mk2<T>(0, 0);
                } else {
                    noise_pair<T>(prm, f, q0 + p2, n0, n1);
                    if (!FULL) {
                        if (2 * p2 >= nvalid) n0 = mk2<T>(0, 0);
                        if (2 * p2 + 1 >= nvalid) n1 = mk2<T>(0, 0);
                    }
                }
                pn2 = csq_acc(n0, pn2);
                if (FULL || 2 * p2 < B) nb[2 * p2] = n0;
                if (2 * p2 + 1 < TC) { pn2 = csq_acc(n1, pn2); if (FULL || 2 * p2 + 1 < B) nb[2 * p2 + 1] = n1; }
            }
            // ---- edge outputs 2t, 2t+1 < E = beta + L - 1 of this thread's symbol: direct form, taps in registers
            const int E = beta + L - 1;
            const bool act = slot < S;
            const int se = act ? slot : S - 1;
            const int ebase = se * stride;
            C2 re0 = mk2<T>(0, 0), re1 = mk2<T>(0, 0);
            {
                C2 h[LB];
#pragma unroll
                for (int l = 0; l < LB; ++l) h[l] = taps[l];
                const C2* src = ub + ebase + 2 * t - (LB - 1);
#pragma unroll
                for (int c = 0; c <= LB; ++c) {
                    const C2 x = src[c];
                    if (c < LB) cmac(re0, h[LB - 1 - c], x);
                    if (c >= 1) cmac(re1, h[LB - c], x);
                }
            }
            const bool e0 = act && 2 * t < E, e1 = act && 2 * t + 1 < E;
            if (!e0) re0 = mk2<T>(0, 0);
            if (!e1) re1 = mk2<T>(0, 0);
            pr2 = csq_acc(re0, pr2);
            pr2 = csq_acc(re1, pr2);
            // ---- interior: c[m], m = t + q*TPF, sits at i = m + cp (and at i -+ N inside the prefix / suffix) if E <= i < stride
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int i = t + q * TPF + cp;
                bool mid = act;
                if (q < ER) mid = mid && i >= E;
                if (q >= 16 - ER) mid = mid && i < stride;
                C2 cq = mid ? cv[q] : mk2<T>(0, 0);
                pr2 = csq_acc(cq, pr2);
                if (q >= 16 - ER) { if (act && i - N >= E) pr2 = csq_acc(cv[q], pr2); }
                if (q < ER) { if (act && i + N < stride) pr2 = csq_acc(cv[q], pr2); }
            }
            if (prm.noise_norm == 1) {
                // the L-1+beta samples the reference truncates still count in both power sums
                // (signal part on the first threads, noise part on the last ones: two warps share the extra latency)
                for (int i = sec + tid; i < body + L - 1; i += NT) pr2 = csq_acc(tail_output<T, LB>(taps, ub, i, body), pr2);
                for (int i = sec + (NT - 1 - tid); i < body + L - 1; i += NT) {
                    C2 n0;
                    if constexpr (VERIFY) n0 = to_v2<T>(prm.noise_in[(size_t)f * prm.noise_len + i]);
                    else n0 = noise_at<T>(prm, f, i);
                    pn2 = csq_acc(n0, pn2);
                }
            }
            T pr = warp_sum(pr2.x + pr2.y), pn = warp_sum(pn2.x + pn2.y);
            if ((tid & 31) == 0) { red[tid >> 5] = pr; red[32 + (tid >> 5)] = pn; }
            __syncthreads();                       // also: every read of the Tx stream is done
            const T g = noise_gain(block_total<NT / 32>(red), snr_lin, block_total<NT / 32>(red + 32));
            // ---- y = r + g n over the stream (noise loads ahead of the may-alias stores)
            const C2* const nz = rbuf + ebase;     // noise by stream position
            {
                C2 y[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) y[q] = caxpy(g, nz[t + q * TPF + cp], cv[q]);
                C2 ye0 = caxpy(g, nz[2 * t], re0), ye1 = caxpy(g, nz[2 * t + 1], re1);
                C2 yp[ER], ys[ER];
#pragma unroll
                for (int q = 0; q < ER; ++q) {
                    const int ip = t + (16 - ER + q) * TPF + cp - N, is = t + q * TPF + cp + N;
                    yp[q] = caxpy(g, nz[max(ip, 0)], cv[16 - ER + q]);
                    ys[q] = caxpy(g, nz[min(is, stride - 1)], cv[q]);
                }
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int i = t + q * TPF + cp;
                    bool mid = act;
                    if (q < ER) mid = mid && i >= E;
                    if (q >= 16 - ER) mid = mid && i < stride;
                    if (mid) ub[ebase + i] = y[q];
                }
#pragma unroll
                for (int q = 0; q < ER; ++q) {
                    const int ip = t + (16 - ER + q) * TPF + cp - N, is = t + q * TPF + cp + N;
                    if (act && ip >= E) ub[ebase + ip] = yp[q];
                    if (act && is < stride) ub[ebase + is] = ys[q];
                }
                if (e0) ub[ebase + 2 * t] = ye0;
                if (e1) ub[ebase + 2 * t + 1] = ye1;
            }
        } else if constexpr (REGS) {
            // Each thread owns the B = prm.chunk stream samples [i0, i0+B).  Their convolution outputs stay
            // in registers across the frame-wide power reduction; their noise is generated INSIDE the
            // convolution loop (one Philox pair every few inputs: integer/MUFU work fills the issue slots
            // the 2-cycle FFMA2s leave free) and parked in shared memory until the gain is known.
            const int B = prm.chunk;
            const int i0 = tid * B;
            const int nvalid = FULL ? TC : min(B, max(sec - i0, 0));
            C2 acc[TC], h[LB];
#pragma unroll
            for (int o = 0; o < TC; ++o) acc[o] = mk2<T>(0, 0);
#pragma unroll
            for (int l = 0; l < LB; ++l) h[l] = taps[l];
            const C2* src = ub + i0 - (LB - 1);
            C2* const nb = rbuf + i0;
            constexpr int NPAIR = (TC + 1) / 2, NSTEP = (TC + LB - 1) / NPAIR;
            const uint32_t q0 = (uint32_t)(rank * NT + tid) * (uint32_t)((B + 1) >> 1);   // block g starts at draw g*(B+1)
            // input c feeds output o through tap (LB-1) - (c - o), 0 <= c - o <= LB-1
#pragma unroll
            for (int c = 0; c < TC + LB - 1; ++c) {
                const C2 x = src[c];
#pragma unroll
                for (int o = 0; o < TC; ++o)
                    if (c - o >= 0 && c - o <= LB - 1) cmac(acc[o], h[LB - 1 - (c - o)], x);
                if (c % NSTEP == 0 && c / NSTEP < NPAIR) {
                    const int p2 = c / NSTEP;
                    C2 n0, n1;
                    if constexpr (VERIFY) {
                        const double2* nin = prm.noise_in + (size_t)f * prm.noise_len + (size_t)rank * sec + i0;
                        n0 = (2 * p2 < nvalid) ? to_v2<T>(nin[2 * p2]) : mk2<T>(0, 0);
                        n1 = (2 * p2 + 1 < nvalid) ? to_v2<T>(nin[2 * p2 + 1]) : mk2<T>(0, 0);
                    } else {
                        noise_pair<T>(prm, f, q0 + p2, n0, n1);
                        if (!FULL) {
                            if (2 * p2 >= nvalid) n0 = mk2<T>(0, 0);
                            if (2 * p2 + 1 >= nvalid) n1 = mk2<T>(0, 0);
                        }
                    }
                    // (slots >= B belong to the next thread's block: never written from here)
                    pn2 = csq_acc(n0, pn2);
                    if (FULL || 2 * p2 < B) nb[2 * p2] = n0;
                    if (2 * p2 + 1 < TC) { pn2 = csq_acc(n1, pn2); if (FULL || 2 * p2 + 1 < B) nb[2 * p2 + 1] = n1; }
                }
            }
            if (!FULL) {
#pragma unroll
                for (int o = 0; o < TC; ++o)
                    if (o >= nvalid) acc[o] = mk2<T>(0, 0);
            }
#pragma unroll
            for (int o = 0; o < TC; ++o) pr2 = csq_acc(acc[o], pr2);
            if (prm.noise_norm == 1 && last_rank) {
                // the L-1+beta samples the reference truncates still count in both power sums
                // (signal part on the first threads, noise part on the last ones: two warps share the extra latency)
                for (int i = sec + tid; i < body + L - 1; i += NT) pr2 = csq_acc(tail_output<T, LB>(taps, ub, i, body), pr2);
                for (int i = sec + (NT - 1 - tid); i < body + L - 1; i += NT) {
                    C2 n0;
                    if constexpr (VERIFY) n0 = to_v2<T>(prm.noise_in[(size_t)f * prm.noise_len + (size_t)rank * sec + i]);
                    else n0 = noise_at<T>(prm, f, rank * sec + i);   // (same numbering: noise_at splits at prm.split = sec)
                    pn2 = csq_acc(n0, pn2);
                }
            }
            // frame-wide sums
            T pr = warp_sum(pr2.x + pr2.y), pn = warp_sum(pn2.x + pn2.y);
            if ((tid & 31) == 0) {
                // warp partials go to slot rank*NW + warp of EVERY CTA of the frame: same order, same gain everywhere
                const int sl = rank * (NT / 32) + (tid >> 5);
#pragma unroll
                for (int r = 0; r < CL; ++r) {
                    T* rr = red;
                    if constexpr (CL > 1) rr = cooperative_groups::this_cluster().map_shared_rank(red, r);
                    rr[sl] = pr; rr[32 + sl] = pn;
                }
            }
            frame_sync<CL>();                      // also: every conv read of the stream is done
            const T g = noise_gain(block_total<CL * (NT / 32)>(red), snr_lin, block_total<CL * (NT / 32)>(red + 32));
            // loads first, then stores: ptxas cannot prove that nb and ub do not overlap and would otherwise
            // serialise every load behind the previous store
#pragma unroll
            for (int o = 0; o < TC; ++o) acc[o] = caxpy(g, nb[o], acc[o]);   // (o >= nvalid: reads a neighbour's slot, result discarded)
#pragma unroll
            for (int o = 0; o < TC; ++o)
                if (FULL || o < nvalid) ub[i0 + o] = acc[o];
        } else {
            const int total = prm.noise_norm == 1 ? body + L - 1 : sec;
            for (int i = tid; i < total; i += NT) {
                C2 a = mk2<T>(0, 0);
                for (int l = 0; l < L; ++l)
                    if (i - l < body) cmac(a, taps[l], ub[i - l]);
                if (i < sec) rbuf[i] = a;
                C2 n0;
                if constexpr (VERIFY) n0 = to_v2<T>(prm.noise_in[(size_t)f * prm.noise_len + i]);
                else n0 = noise_at<T>(prm, f, i);
                pr2 = csq_acc(a, pr2);
                pn2 = csq_acc(n0, pn2);
            }
            T pr = warp_sum(pr2.x + pr2.y), pn = warp_sum(pn2.x + pn2.y);
            if ((tid & 31) == 0) { red[tid >> 5] = pr; red[32 + (tid >> 5)] = pn; }
            __syncthreads();
            const T g = noise_gain(block_total<NT / 32>(red), snr_lin, block_total<NT / 32>(red + 32));
            for (int i = tid; i < sec; i += NT) {
                C2 n0;
                if constexpr (VERIFY) n0 = to_v2<T>(prm.noise_in[(size_t)f * prm.noise_len + i]);
                else n0 = noise_at<T>(prm, f, i);
                ub[i] = caxpy(g, n0, rbuf[i]);
            }
        }
        __syncthreads();

        // =========================== receiver ===========================
        // block s: z[k] = wrx[k]*y[s*stride + rm + k]; o[n] = sum_{k = n + hh (mod N)} z[k];
        // q[n] = o[(n + shift) mod N]; Y = DFT(q)   (receiver.py:13-133)
        unsigned bit_cnt = 0, sym_cnt = 0;
        for (int s0 = 0; s0 < S; s0 += FPP) {
            const int s = s0 + slot;
            const bool act = s < S;
            const int se = act ? s : S - 1;
            C2 v[16];
            const C2* ys = ub + se * stride + prm.rm + hh;
            const T* wr = wrx + hh;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                if (REGS && q >= 1 && q <= 13) {
                    // tail_rx/2, shift <= TPF: rows 1..13 neither wrap nor touch the overlap-add margins
                    const int n = t + q * TPF + prm.shift;
                    v[q] = cscale(wr[n], ys[n]);
                    continue;
                }
                const int a0 = (q * TPF + prm.shift) & (N - 1);          // first n of this register row
                const int n = (t + q * TPF + prm.shift) & (N - 1);
                C2 o = cscale(wr[n], ys[n]);
                if (hh > 0) {                                             // uniform
                    const bool wraps = a0 + TPF > N;
                    if (wraps || a0 < hh) { if (n < hh) o = caxpy(wr[n + N], ys[n + N], o); }
                    if (wraps || a0 + TPF > N - hh) { if (n >= N - hh) o = caxpy(wr[n - N], ys[n - N], o); }
                }
                v[q] = o;
            }
            fft_regs<T, N, -1, FPP>(v, t, xb, tw, slot);
            const uint4 wv = symw[se * TPF + t];
            const uint32_t w[4] = {wv.x, wv.y, wv.z, wv.w};
            if (s0 == 0) {
                // pilot (wofdm_simulation.py:223): the pilot's threads publish Y0, then every thread turns one
                // bin into the equaliser tap G[k] = X0[k] / Y0[k] (lattice units), so nobody waits on one warp
                if (rank == 0) {
                    if (se == 0) {
#pragma unroll
                        for (int q = 0; q < 16; ++q) geq[t + q * TPF] = v[q];
                    }
                    __syncthreads();
                    const unsigned char* pil = reinterpret_cast<const unsigned char*>(symw);   // symbol 0: thread k%TPF, byte k/TPF
                    for (int k = tid; k < N; k += NT) {
                        const C2 y0 = geq[k];
                        const C2 x0 = qlut[pil[(k % TPF) * 16 + k / TPF]];
                        C2 gk = cscale(recip(y0.x * y0.x + y0.y * y0.y), cmulc(x0, y0));
                        if (prm.guard > 0 && !bin_active<N>(k, prm.guard)) gk = mk2<T>(0, 0);   // null bin: equalised value 0 + 0i
                        geq[k] = gk;
                        if constexpr (CL > 1) {
#pragma unroll
                            for (int r = 1; r < CL; ++r) cooperative_groups::this_cluster().map_shared_rank(geq, r)[k] = gk;
                        }
                    }
                }
                frame_sync<CL>();
            }
            if (act && sb + s > 0) {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int k = t + q * TPF;
                    const C2 e = cmul(v[q], geq[k]);                                       // :231
                    const int dec = slice_index(e, hb);                                    // :233 (level code)
                    const int txi = sym_byte(w, q);
                    sym_cnt += (dec != txi);                                               // :235
                    bit_cnt += code_bit_errors((uint32_t)(dec ^ txi), gxm);
                    if constexpr (RES) { if (prm.res_bins && dec != txi) res_add4(racc, (uint32_t)(dec ^ txi), gxm, k, 0); }
                    if constexpr (VERIFY) {
                        const size_t o = ((size_t)f * (prm.S - 1) + (sb + s - 1)) * N + k;
                        prm.eq_out[o] = make_double2((double)e.x * prm.qscale, (double)e.y * prm.qscale);
                        prm.dec_out[o] = levels_to_idx(dec >> hb, dec & (m - 1), hb, m, prm.constellation);
                    }
                }
            }
        }
        bit_cnt = warp_sum(bit_cnt);
        sym_cnt = warp_sum(sym_cnt);
        if constexpr (RES) {
            if (!prm.res_bins && (tid & 31) == 0) {      // per-cell totals: the per-warp atomics at the cell's address
                atomicAdd(prm.counters + 2 * rcell, (unsigned long long)bit_cnt);
                atomicAdd(prm.counters + 2 * rcell + 1, (unsigned long long)sym_cnt);
            }
        } else if ((tid & 31) == 0) {
            if constexpr (VERIFY) {
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.bit_err_f) + f, (unsigned long long)bit_cnt);
                atomicAdd(reinterpret_cast<unsigned long long*>(prm.sym_err_f) + f, (unsigned long long)sym_cnt);
            } else {
                atomicAdd(prm.counters + 2 * si, (unsigned long long)bit_cnt);
                atomicAdd(prm.counters + 2 * si + 1, (unsigned long long)sym_cnt);
            }
        }
        // the register policy with one CTA per frame needs no barrier here: taps were copied to registers before the power
        // barrier, the stream and the symbol words were last read before the pilot barriers, the parked noise before the
        // receiver's; geq and red are rewritten only behind the next frame's own barriers (CIRC recomputes hf from taps
        // behind its own barriers but reads them late; clusters and the staged policy keep the barrier)
        // (a frame received in more than one pass, S > FPP, reads the stream after the pilot barriers: it keeps the barrier too)
        if (!(REGS && CL == 1 && !CIRC && !VERIFY) || S > FPP) __syncthreads();   // taps / stream / geq are rewritten by the next frame
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
                    __syncthreads();                     // every decision of the cell has been added
                    res_flush(racc, N, N, ncell * N, prm.counters + (size_t)rcell * N * 2, tid, NT);
                    rcell = nc; rfr = 0;
                }
            } else {
                rcell = prm.res_chan ? si * prm.C + ci : si;
            }
        }
    }
    if constexpr (CL > 1) cooperative_groups::this_cluster().sync();   // nobody leaves while a peer may still read its shared memory
}

// ---- export of the on-device draws (wofdm_ber_draws) ------------------------------------------
template <int N>
__global__ void draws_sym_kernel(BerParams prm, const long long* frame_ids, int32_t* out) {
    constexpr int TPF = N / 16;
    const long long f = frame_ids[blockIdx.y];
    const int s = blockIdx.x;
    for (int t = threadIdx.x; t < TPF; t += blockDim.x) {
        uint32_t w[4];
        load_sym_idx<N, false>(prm, f, s, t, w);
        const int hb = prm.bits >> 1, m = 1 << hb;
        for (int q = 0; q < 16; ++q) {
            const int code = sym_byte(w, q);
            out[((size_t)blockIdx.y * prm.S + s) * N + t + q * TPF] = levels_to_idx(code >> hb, code & (m - 1), hb, m, prm.constellation);
        }
    }
}
template <typename T>
__global__ void draws_noise_kernel(BerParams prm, const long long* frame_ids, double2* out) {
    const long long f = frame_ids[blockIdx.y];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // stream position
    if (i >= prm.noise_len) return;
    const V2<T> n0 = noise_at<T>(prm, f, (int)i);
    out[(size_t)blockIdx.y * prm.noise_len + i] = make_double2((double)n0.x, (double)n0.y);
}

}  // namespace wofdm
