// mask_gemm.cu -- Tx side of the channel-mask BER variant (SURVEY.md section 8f-1) as ONE dense product on the 5th-generation
// tensor cores (tcgen05, kind::f16).
//
// matlab/main_channel_mask.m:384-417 builds a masked OFDM symbol by a chain of dense matrices: inverse DFT of the guarded
// symbol vector, redundancy, Tx window (gen_tx_ofdm), then dft_rc_filt: zero-pad to M = 2 n_tx - 1, DFT_M, raised-cosine
// mask, inverse DFT_M.  Every factor is linear and none depends on the data, so the masked symbol is
//
//     y = Mm a,      Mm[r, c] = sum_j g[(r - j) mod M] w_tx[j] exp(2 pi i k_c ((j - cp) mod N) / N)      (M x nact, complex)
//
// with a the nact = N - 2 guard lattice points of the symbol, k_c the bin of active sub-carrier c and g =
// IDFT_M(ifftshift(windowRC)).  mask_kernel.cuh evaluates that chain per symbol with two 8N-point register FFTs (225 kflop
// per symbol at N = 256: three times the whole unmasked chain); here it is the GEMM the reference writes down:
//
//     [Re y; Im y] (2M rows, interleaved) = A (2M x 2 nact, real form of Mm) . [Re a; Im a]  for all symbols of a batch at once.
//
// dft_rc_filt then keeps samples 0..n_tx-1 of y_s in symbol s and adds the other n_tx - 1 to the start of symbol s+1 (:413-416).
// That is linear too and goes into the product's K dimension: with Mm = [Mtop; Mbot] (rows 0..n_tx-1 and n_tx..M-1, a zero row
// appended), the filtered symbol is
//
//     f_s = y_s[0..n_tx) + y_{s-1}[n_tx..M) = [Mtop | Mbot] [a_s; a_{s-1}]          (a_{-1} = 0)
//
// -- the same number of MACs (n_tx x 2 nact instead of M x nact), half the output.  The B operand holds, per column (frame, s),
// the lattice points of symbol s followed by those of symbol s-1.
//
// The lattice points are small odd integers -- exact in fp16 -- and A is split A = hi + lo in fp16 behind a power-of-two
// scale (relative error ~2^-22 per entry, fp32 accumulation in tensor memory): two MMAs per K step give fp32-grade
// results, 1.3 Mflop per symbol (N = 256, 128 active sub-carriers).  Kernels:
//   mask_response_kernel, mask_matrix_kernel, mask_split_kernel   g and Mm in fp64 on the device (once per call), Mm split
//                                            into pre-tiled hi | lo operands
//   mask_sym_kernel                          the Philox symbol draws of K1 (load_sym_idx) -> lattice points as fp16 B tiles
//   mask_gemm_f16                            persistent, warp-specialised: bulk-copy producer, one MMA thread, four epilogue
//                                            warps; two 128 x 256 accumulators in tensor memory, three 64 KB stages
//   mask_assemble_kernel                     (K1 kernels other than ber_tconv2.cuh, which gathers from Y itself:) the filtered
//                                            symbols overlap-added with the frame stride (tx2rx, :420-431): the serialised
//                                            stream K1 reads (BerParams::tx_stream)
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "ber_kernel.cuh"
#include "mask_gemm.h"

namespace wofdm {

namespace {

constexpr int TM = 128, TN = 256, KB = 64, NSTAGE = 3;
constexpr int A_HALVES = TM * KB, B_HALVES = TN * KB;                  // one A (hi or lo) tile, one B tile
constexpr int A_BYTES = A_HALVES * 2, B_BYTES = B_HALVES * 2;
constexpr int STAGE_BYTES = 2 * A_BYTES + B_BYTES;                     // 64 KiB
// D = f32, A = B = f16, both K-major, N = 256, M = 128
constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
constexpr int NTHREADS = 192;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE core matrices (8 rows x 16 bytes): LBO = 128 B between the two K chunks of one MMA, SBO = 1024 B
// between 8-row groups
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((128u >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((1024u >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;                       // descriptor version of sm_100
    return d;
}
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(da), "l"(db), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (int it = 0; it < (1 << 22) && !done; ++it)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done) __trap();                          // never spin forever on a GPU we share
}
__device__ __forceinline__ void bulk_copy(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// offsets (in halves) inside the pre-tiled operands: 16-byte chunk = (row / 8) * 64 + (k / 8) * 8 + row % 8
__host__ __device__ __forceinline__ size_t a_off(int row, int k, int nk) {
    const int rt = row / TM, r = row % TM, kb = k / KB, kk = k % KB;
    return ((size_t)rt * nk + kb) * (2 * (size_t)A_HALVES) + (size_t)(((r >> 3) * 64 + (kk >> 3) * 8 + (r & 7)) * 8 + (kk & 7));
}
__host__ __device__ __forceinline__ size_t b_off(long long col, int k, int nk) {
    const long long ct = col / TN;
    const int c = (int)(col % TN), kb = k / KB, kk = k % KB;
    return ((size_t)ct * nk + kb) * (size_t)B_HALVES + (size_t)(((c >> 3) * 64 + (kk >> 3) * 8 + (c & 7)) * 8 + (kk & 7));
}

// g = IDFT_M(ifftshift(windowRC)) (main_channel_mask.m:404-412; gen_raised_cosine :477-493): thread = one sample
__global__ void __launch_bounds__(64) mask_response_kernel(double2* __restrict__ g, int M, int roll_off) {
    extern __shared__ double wsh[];                        // ifftshift(windowRC) [M], then the phasors exp(2 pi i m / M) [2 M]
    double* const phc = wsh + M;
    double* const phs = phc + M;
    const int wl = M / 2, rest = M - wl - 2 * roll_off, zl = rest / 2;
    for (int k = threadIdx.x; k < M; k += blockDim.x) {
        sincospi(2.0 * (double)k / (double)M, &phs[k], &phc[k]);
        const int i = (k + M / 2) % M - zl;                // position inside [raised cosine | ones | falling cosine]
        double w = 0.0;
        if (i >= 0 && i < 2 * roll_off + wl) {
            const int e = i < roll_off ? i : i >= roll_off + wl ? 2 * roll_off + wl - 1 - i : -1;
            if (e < 0) w = 1.0;
            else {
                double sn, cs;
                sincospi(0.5 * (0.5 + (-(roll_off + 1) / 2.0 + 1.0 + e) / roll_off), &sn, &cs);
                w = sn * sn;
            }
        }
        wsh[k] = w;
    }
    __syncthreads();
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= M) return;
    double re = 0.0, im = 0.0;
    int idx = 0;                                           // k n mod M
    for (int k = 0; k < M; ++k) {
        const double w = wsh[k];
        re += w * phc[idx]; im += w * phs[idx];
        idx += n;
        if (idx >= M) idx -= M;
    }
    g[n] = make_double2(re / M, im / M);
}

// Mm[r][c] in fp64: thread = one entry, the phasors exp(2 pi i m / N) from a shared table
__global__ void __launch_bounds__(256) mask_matrix_kernel(const double2* __restrict__ g, const float* __restrict__ wtx, double2* __restrict__ Mm,
                                                          unsigned* __restrict__ maxbits, int N, int n_tx, int cp, int guard, int M, int nact) {
    extern __shared__ double2 ph[];
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        double s, c;
        sincospi(2.0 * (double)i / (double)N, &s, &c);
        ph[i] = make_double2(c, s);
    }
    __syncthreads();
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= M * nact) return;
    const int r = e / nact, c = e % nact;
    const int bin = (c + guard + N / 2) & (N - 1);         // bin_active (ber_kernel.cuh): centred index c + guard
    double re = 0.0, im = 0.0;
    int gi = r;                                            // (r - j) mod M
    for (int j = 0; j < n_tx; ++j) {
        const double2 p = ph[(bin * ((j - cp) & (N - 1))) & (N - 1)];
        const double w = (double)wtx[j];
        const double2 gv = g[gi];
        re += w * (gv.x * p.x - gv.y * p.y);
        im += w * (gv.x * p.y + gv.y * p.x);
        gi = gi == 0 ? M - 1 : gi - 1;
    }
    Mm[e] = make_double2(re, im);
    atomicMax(maxbits, __float_as_uint((float)fmax(fabs(re), fabs(im))));
}

// real form, scaled by a power of two into the comfortable fp16 range and split hi + lo, straight into the UMMA tiles:
// A[2r][2c] = Re, A[2r][2c+1] = -Im, A[2r+1][2c] = Im, A[2r+1][2c+1] = Re of Mm[r][c] in columns [0, Kp/2) (r < n_tx: Mtop) and of
// Mm[n_tx + r][c] in columns [Kp/2, Kp) (Mbot); rows >= 2 n_tx, row n_tx - 1 of Mbot and the K padding are zero
__global__ void __launch_bounds__(256) mask_split_kernel(const double2* __restrict__ Mm, const unsigned* __restrict__ maxbits, __half* __restrict__ At,
                                                         float* __restrict__ scale_out, int M, int n_tx, int nact, int Kp, int RT) {
    const float mx = __uint_as_float(*maxbits);
    const int ex = mx > 0.f ? 11 - ilogbf(mx) : 0;         // largest entry lands in [2^11, 2^12)
    const double sc = ldexp(1.0, ex);
    if (blockIdx.x == 0 && threadIdx.x == 0) { scale_out[0] = (float)sc; scale_out[1] = (float)ldexp(1.0, -ex); }
    const int nk = Kp / KB;
    const size_t total = (size_t)RT * TM * Kp;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int R = (int)(i / Kp), k = (int)(i % Kp);
        double x = 0.0;
        const int part = k >= Kp / 2, kk = k - part * (Kp / 2), row = (R >> 1) + part * n_tx;
        if (R < 2 * n_tx && row < M && kk < 2 * nact) {
            const double2 v = Mm[(size_t)row * nact + (kk >> 1)];
            x = (R & 1) ? ((kk & 1) ? v.x : v.y) : ((kk & 1) ? -v.y : v.x);
        }
        x *= sc;
        const __half hi = __float2half_rn((float)x);
        const __half lo = __float2half_rn((float)(x - (double)__half2float(hi)));
        const size_t o = a_off(R, k, nk);
        At[o] = hi;
        At[o + A_HALVES] = lo;
    }
}

// the symbols of the batch, exactly as K1 draws them (load_sym_idx): one CTA per frame; thread (s, t) holds the 16 level codes
// of bins t + q TPF and parks the lattice points of the active ones, (Re, Im) fp16 pairs, in shared memory; the frame's columns
// then leave as 16-byte chunks (four sub-carriers; consecutive lanes = consecutive columns of a core matrix): into the first
// half of column frame * S + s (a_s) and into the second half of the next symbol's column (a_{s-1} there; symbol 0's second
// half stays zero).  SEG: f0 + fl is a local index into the segment table draw.seg, decoded by seg_frame.
template <int N, bool SEG = false>
__global__ void __launch_bounds__(256) mask_sym_kernel(const BerParams draw, long long f0, long long nf, int S, int guard, int nact,
                                                       __half* __restrict__ Bt, int nk) {
    constexpr int TPF = N / 16;
    extern __shared__ __align__(16) __half2 lat[];         // [S][rowp]
    const int khalf = nk * KB / 2;
    const int hb = draw.bits >> 1, m = 1 << hb;
    const int nchunk = (nact + 3) / 4, rowp = 4 * nchunk + 4;
    for (int e = threadIdx.x; e < S * rowp; e += blockDim.x) lat[e] = __floats2half2_rn(0.f, 0.f);
    __syncthreads();
    for (long long fl = blockIdx.x; fl < nf; fl += gridDim.x) {
        long long f = f0 + fl;
        if constexpr (SEG) { int si, ci; seg_frame(draw, f, f, si, ci); }
        for (int e = threadIdx.x; e < S * TPF; e += blockDim.x) {
            const int s = e / TPF, t = e % TPF;
            uint32_t w[4];
            load_sym_idx<N, false>(draw, f, s, t, w);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int bin = t + q * TPF;
                const int c = ((bin + N / 2) & (N - 1)) - guard;
                if (c >= 0 && c < nact) {
                    const int code = sym_byte(w, q);
                    lat[s * rowp + c] = __floats2half2_rn((float)(2 * (code >> hb) - (m - 1)), (float)(2 * (code & (m - 1)) - (m - 1)));
                }
            }
        }
        __syncthreads();
        for (int e = threadIdx.x; e < S * nchunk; e += blockDim.x) {
            const int s = e % S, kc = e / S;
            const uint4 v = *reinterpret_cast<const uint4*>(lat + s * rowp + 4 * kc);
            const long long col = fl * S + s;
            *reinterpret_cast<uint4*>(Bt + b_off(col, 8 * kc, nk)) = v;
            if (s + 1 < S) *reinterpret_cast<uint4*>(Bt + b_off(col + 1, khalf + 8 * kc, nk)) = v;
        }
        __syncthreads();
    }
}

// Persistent: CTA q takes the tiles q, q + grid, ...; tile p = (column tile p / RT, row tile p % RT) -- CTAs that run side by
// side share their B tile in L2.  Warps 0-3 = epilogue (TMEM lanes 32w..32w+31), warp 4 = producer, warp 5 = MMA issuer.
__global__ void __launch_bounds__(NTHREADS, 1) mask_gemm_f16(const __half* __restrict__ At, const __half* __restrict__ Bt, float* __restrict__ Y,
                                                            const float* __restrict__ scale, int nk, int RT, int n_tiles, int Yp, long long ncols) {
    extern __shared__ __align__(1024) unsigned char sm[];
    __shared__ __align__(8) unsigned long long full_bar[NSTAGE], empty_bar[NSTAGE], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (warp == 4) {   // both accumulators: all 512 columns (one CTA per SM: the stages take 192 KB of shared memory)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(2 * TN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < NSTAGE; ++i) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&full_bar[i])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&empty_bar[i])) : "memory");
        }
        for (int i = 0; i < 2; ++i) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&acc_full[i])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" :: "r"(smem_u32(&acc_empty[i])) : "memory");   // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    if (warp == 4) {
        if (lane == 0) {
            // ===== producer: two bulk copies per stage (A hi | lo, B), K blocks numbered through all of this CTA's tiles =====
            int it = 0;
            for (int p = blockIdx.x; p < n_tiles; p += gridDim.x) {
                const __half* ra = At + (size_t)(p % RT) * nk * (2 * (size_t)A_HALVES);
                const __half* rb = Bt + (size_t)(p / RT) * nk * (size_t)B_HALVES;
                for (int kb = 0; kb < nk; ++kb, ++it) {
                    const int st = it % NSTAGE;
                    if (it >= NSTAGE) mbar_wait(smem_u32(&empty_bar[st]), (uint32_t)(((it / NSTAGE) - 1) & 1));
                    const uint32_t bar = smem_u32(&full_bar[st]), dst = smem_u32(sm + (size_t)st * STAGE_BYTES);
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"((uint32_t)STAGE_BYTES) : "memory");
                    bulk_copy(dst, ra + (size_t)kb * (2 * (size_t)A_HALVES), 2 * A_BYTES, bar);
                    bulk_copy(dst + 2 * A_BYTES, rb + (size_t)kb * (size_t)B_HALVES, B_BYTES, bar);
                }
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {
            // ===== MMA issuer: tile tl accumulates into TMEM columns [(tl & 1) * TN, +TN) while the epilogue drains the other half =====
            int it = 0, tl = 0;
            for (int p = blockIdx.x; p < n_tiles; p += gridDim.x, ++tl) {
                const int buf = tl & 1;
                if (tl >= 2) {
                    mbar_wait(smem_u32(&acc_empty[buf]), (uint32_t)(((tl >> 1) - 1) & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                const uint32_t tacc = tmem + (uint32_t)(buf * TN);
                for (int kb = 0; kb < nk; ++kb, ++it) {
                    const int st = it % NSTAGE;
                    mbar_wait(smem_u32(&full_bar[st]), (uint32_t)((it / NSTAGE) & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_hi = smem_u32(sm + (size_t)st * STAGE_BYTES), a_lo = a_hi + A_BYTES, b = a_hi + 2 * A_BYTES;
#pragma unroll
                    for (int j = 0; j < KB / 16; ++j) {                            // one MMA consumes 16 halves = two 16-byte chunks
                        const uint32_t off = (uint32_t)j * 256u;
                        mma_f16(tacc, umma_desc(a_hi + off), umma_desc(b + off), (kb | j) != 0);
                        mma_f16(tacc, umma_desc(a_lo + off), umma_desc(b + off), 1u);
                    }
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(&empty_bar[st])) : "memory");
                }
                // completes once per tile, after every MMA of the tile
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(&acc_full[buf])) : "memory");
            }
        }
    } else {
        // ===== epilogue warps: thread = one row of the tile (TMEM lane 32 warp + lane): for every column (symbol) the warp
        //       stores 32 consecutive floats of Y =====
        const float descale = scale[1];
        int tl = 0;
        for (int p = blockIdx.x; p < n_tiles; p += gridDim.x, ++tl) {
            const int buf = tl & 1;
            const long long col0 = (long long)(p / RT) * TN;
            const int r = (p % RT) * TM + warp * 32 + lane;
            mbar_wait(smem_u32(&acc_full[buf]), (uint32_t)((tl >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float* yrow = Y + (size_t)col0 * Yp + r;
#pragma unroll 1
            for (int cc = 0; cc < TN / 32; ++cc) {
                uint32_t v[32];
                const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * TN + cc * 32);
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                      "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                      "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                    : "r"(taddr) : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (col0 + cc * 32 < ncols) {                                   // (columns behind the batch: nobody reads them)
#pragma unroll
                    for (int i = 0; i < 32; ++i) yrow[(size_t)(cc * 32 + i) * Yp] = __uint_as_float(v[i]) * descale;
                }
            }
            // this warp's quarter of the accumulator has been read: hand the buffer back to the MMA issuer
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(&acc_empty[buf])) : "memory");
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(2 * TN) : "memory");
}

// stream[f][p], p = s stride + i: the filtered symbols (columns of Y) overlap-added with the frame stride,
// stream[s stride + i] = f_s[i] + f_{s-1}[stride + i] (the second term while stride + i < n_tx; s = S: the last symbol's tail)
__global__ void __launch_bounds__(256) mask_assemble_kernel(const float* __restrict__ Y, float2* __restrict__ stream, long long nf, int S, int stride,
                                                            int n_tx, int tail_tx, int Yp) {
    const int body = tail_tx + S * stride;
    const long long total = nf * body;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long fl = e / body;
        const int p = (int)(e - fl * body);
        const int s = min(p / stride, S), i = p - s * stride;
        const float* ys = Y + (size_t)(fl * S + s) * Yp;
        float2 a = make_float2(0.f, 0.f), c = make_float2(0.f, 0.f);
        if (s < S) a = *reinterpret_cast<const float2*>(ys + 2 * i);
        if (s >= 1 && stride + i < n_tx) c = *reinterpret_cast<const float2*>(ys - Yp + 2 * (stride + i));
        stream[e] = cadd(a, c);
    }
}

}  // namespace

size_t mask_gemm_plan(const wofdm_sys_t& sys, long long batch, MaskGemm& mg) {
    memset(&mg, 0, sizeof(mg));
    mg.N = sys.N; mg.S = sys.S; mg.cp = sys.cp; mg.bits = sys.bits; mg.guard = sys.guard; mg.tail_tx = sys.tail_tx;
    mg.n_tx = sys.N + sys.cp + sys.cs; mg.stride = mg.n_tx - sys.tail_tx; mg.M = 2 * mg.n_tx - 1;
    mg.nact = sys.N - 2 * sys.guard;
    mg.Kp = 2 * ((2 * mg.nact + KB - 1) / KB * KB); mg.nk = mg.Kp / KB;          // [a_s | a_{s-1}], each half padded to the K block
    mg.RT = (2 * mg.n_tx + TM - 1) / TM; mg.Yp = mg.RT * TM;
    mg.batch = batch;
    const size_t cols = (size_t)((batch * sys.S + TN - 1) / TN) * TN;
    return (size_t)mg.RT * mg.nk * 2 * A_BYTES + cols * mg.Kp * 2 + cols * mg.Yp * 4 + (size_t)mg.M * 16 + (size_t)mg.M * mg.nact * 16 + 4096;
}

int mask_gemm_setup(wofdm_ctx* h, DeviceCtx& d, MaskGemm& mg, int roll_off, const float* d_wtx) {
    const size_t cols = (size_t)((mg.batch * mg.S + TN - 1) / TN) * TN;
    const size_t at_b = (size_t)mg.RT * mg.nk * 2 * A_BYTES, bt_b = cols * mg.Kp * 2, y_b = cols * mg.Yp * 4;
    mg.At = static_cast<__half*>(arena_take(d, at_b));
    mg.Bt = static_cast<__half*>(arena_take(d, bt_b));
    mg.Y = static_cast<float*>(arena_take(d, y_b));
    mg.g = static_cast<double2*>(arena_take(d, (size_t)mg.M * 16));
    mg.Mm = static_cast<double2*>(arena_take(d, (size_t)mg.M * mg.nact * 16));
    mg.scale = static_cast<float*>(arena_take(d, 16));
    mg.maxbits = static_cast<unsigned*>(arena_take(d, 16));
    if (!mg.At || !mg.Bt || !mg.Y || !mg.g || !mg.Mm || !mg.scale || !mg.maxbits) return fail(h, WOFDM_ENOMEM, "mask product: arena exhausted");
    mask_response_kernel<<<(mg.M + 63) / 64, 64, (size_t)mg.M * 24, d.stream>>>(mg.g, mg.M, roll_off);
    WOFDM_CUDA(h, cudaGetLastError());
    WOFDM_CUDA(h, cudaMemsetAsync(mg.maxbits, 0, 4, d.stream));
    WOFDM_CUDA(h, cudaMemsetAsync(mg.Bt, 0, bt_b, d.stream));      // K padding and the columns behind the batch stay zero
    const int ne = mg.M * mg.nact;
    mask_matrix_kernel<<<(ne + 255) / 256, 256, (size_t)mg.N * 16, d.stream>>>(mg.g, d_wtx, mg.Mm, mg.maxbits, mg.N, mg.n_tx, mg.cp, mg.guard, mg.M, mg.nact);
    WOFDM_CUDA(h, cudaGetLastError());
    mask_split_kernel<<<2 * d.sm_count, 256, 0, d.stream>>>(mg.Mm, mg.maxbits, mg.At, mg.scale, mg.M, mg.n_tx, mg.nact, mg.Kp, mg.RT);
    WOFDM_CUDA(h, cudaGetLastError());
    WOFDM_CUDA(h, cudaFuncSetAttribute(mask_gemm_f16, cudaFuncAttributeMaxDynamicSharedMemorySize, NSTAGE * STAGE_BYTES));
    h->launches += 3;
    return WOFDM_OK;
}

int mask_gemm_batch(wofdm_ctx* h, DeviceCtx& d, const MaskGemm& mg, uint64_t seed, long long f0, long long nf, float2* stream,
                    const long long* seg, int n_seg, int C, long long ensemble) {
    if (nf < 1 || nf > mg.batch) return fail(h, WOFDM_EINVAL, "mask product: batch out of range");
    BerParams draw;
    memset(&draw, 0, sizeof(draw));
    draw.seed = seed; philox_round_keys(seed, draw.rk); draw.bits = mg.bits; draw.S = mg.S;
    draw.C = C; draw.ensemble = ensemble; draw.seg = seg; draw.n_seg = n_seg;
    const long long ncols = nf * mg.S;
    const int grid_s = (int)std::min<long long>(nf, (long long)d.sm_count * 8);
    const size_t sm_s = (size_t)mg.S * (4 * ((mg.nact + 3) / 4) + 4) * sizeof(__half2);
    if (sm_s > d.smem_optin) return fail(h, WOFDM_EUNSUPPORTED, "mask product: too many symbols per frame for the symbol kernel");
    using SymFn = void (*)(const BerParams, long long, long long, int, int, int, __half*, int);
    SymFn fn = nullptr;
    switch (mg.N) {
        case 128: fn = seg ? mask_sym_kernel<128, true> : mask_sym_kernel<128>; break;
        case 256: fn = seg ? mask_sym_kernel<256, true> : mask_sym_kernel<256>; break;
        case 512: fn = seg ? mask_sym_kernel<512, true> : mask_sym_kernel<512>; break;
        default: return fail(h, WOFDM_EUNSUPPORTED, "the channel-mask variant is built for N = 128, 256, 512");
    }
    if (sm_s > 48 * 1024)                   // (long frames: more than the default dynamic shared memory)
        WOFDM_CUDA(h, cudaFuncSetAttribute((const void*)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_s));
    fn<<<grid_s, 256, sm_s, d.stream>>>(draw, f0, nf, mg.S, mg.guard, mg.nact, mg.Bt, mg.nk);
    WOFDM_CUDA(h, cudaGetLastError());
    const int CT = (int)((ncols + TN - 1) / TN), n_tiles = CT * mg.RT;
    mask_gemm_f16<<<std::min(n_tiles, d.sm_count), NTHREADS, NSTAGE * STAGE_BYTES, d.stream>>>(mg.At, mg.Bt, mg.Y, mg.scale, mg.nk, mg.RT, n_tiles, mg.Yp, ncols);
    WOFDM_CUDA(h, cudaGetLastError());
    h->launches += 2;
    if (!stream) return WOFDM_OK;          // (the K1 kernel gathers from Y itself: ber_tconv2.cuh, tconv2_load_masked)
    const long long total = nf * (mg.tail_tx + (long long)mg.S * mg.stride);
    mask_assemble_kernel<<<(int)std::min<long long>((total + 255) / 256, (long long)d.sm_count * 16), 256, 0, d.stream>>>(
        mg.Y, stream, nf, mg.S, mg.stride, mg.n_tx, mg.tail_tx, mg.Yp);
    WOFDM_CUDA(h, cudaGetLastError());
    h->launches += 1;
    return WOFDM_OK;
}

}  // namespace wofdm
