// interf.cu -- K2/K3: interference power of the w-OFDM systems over every channel realisation.
//
//   A_m(c) = Rx_mat . H_m(h_c) . Tx_mat,   P_k(c) = sum_{j != k} |A_0[k,j]|^2 + sum_{m>=1} sum_j |A_m[k,j]|^2
//
// replacing interf_power (python/ofdm_utils/interf_calc.py:20-113) and calculate_interference
// (matlab/main_interference_calculation.m:177-225), which evaluate ONE (mean) channel with eight dense
// N x n products per A matrix.  Here:
//   K3  build_tx_matrix / build_rx_matrix: Tx_mat = Vtx.Gamma.W^-1 (n_tx x N) and Rx_mat = W.K.P.Vrx.R
//       (N x n_rx) written in closed form (one sincospi per entry) -- the matrix builders of
//       transmitter.py / receiver.py / matlab/functions/*_matrix.m.
//   K2a build_b: B_m(c) = H_m(h_c).Tx_mat.  H_m is banded Toeplitz (channel.py:15-53), so this is an
//       L-tap convolution down the columns of Tx_mat; written to HBM as the real matrix [Re B; Im B].
//   K2b gemm_power_f64: the dense contraction [Re A; Im A] = [Rr -Ri; Ri Rr] . [Re B; Im B] on the FP64
//       tensor path (mma.sync m8n8k4 f64 = DMMA), all channels and slices side by side as the N
//       dimension, with the off-diagonal mask and the row-wise sum of |.|^2 fused into the epilogue.
// The TF32-split tensor path (mode 1) lives in interf_tf32.cu.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <type_traits>

#include "host_common.h"
#include "interf.h"

namespace wofdm {

// ---- K3: matrix builders ----------------------------------------------------------------------
// Tx_mat[i][k] = vtx[i]/N * exp(+2 pi i k n / N), n = (i - cp) mod N      (transmitter.py:13-58)
// (T32, optional: the same matrix rounded to fp32 for the TF32 path's band product)
__global__ void build_tx_matrix(double2* __restrict__ T, const double* __restrict__ vtx, int N, int cp, int n_tx,
                                float2* __restrict__ T32 = nullptr) {
    const int i = blockIdx.x, n = ((i - cp) % N + N) % N;
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
        double s, c;
        sincospi(2.0 * (double)(((long long)k * n) % N) / (double)N, &s, &c);
        const double w = vtx[i] / (double)N;
        T[(size_t)i * N + k] = make_double2(w * c, w * s);
        if (T32) T32[(size_t)i * N + k] = make_float2((float)(w * c), (float)(w * s));
    }
}

// Rbig (2N x Kp), the real form of Rx_mat with the K dimension INTERLEAVED: column 2b multiplies Re B[b], column
// 2b+1 multiplies Im B[b] (so the non-zero rows of an ISI slice are a prefix of K, see build_b):
//   row k   (Re A): [ Rr[k][b], -Ri[k][b] ],   row N+k (Im A): [ Ri[k][b], Rr[k][b] ]
// R[k][b] = vrx[b-rm] * exp(-2 pi i k n(b) / N) for rm <= b < rm+N+d, n(b) = ((b - rm - d/2) mod N - shift) mod N
//                                                                                          (receiver.py:13-133)
__global__ void build_rx_matrix(double* __restrict__ Rbig, const double* __restrict__ vrx, int N, int tail_rx,
                                int rm, int shift, int n_rx, int Kp) {
    const int k = blockIdx.x;
    const int hh = tail_rx / 2;
    for (int b = threadIdx.x; 2 * b < Kp; b += blockDim.x) {
        double re = 0.0, im = 0.0;
        if (b < n_rx && b >= rm && b - rm < N + tail_rx) {
            const int np = ((b - rm - hh) % N + N) % N;
            const int n = ((np - shift) % N + N) % N;
            double s, c;
            sincospi(2.0 * (double)(((long long)k * n) % N) / (double)N, &s, &c);
            re = vrx[b - rm] * c;
            im = -vrx[b - rm] * s;
        }
        *reinterpret_cast<double2*>(Rbig + (size_t)k * Kp + 2 * b) = make_double2(re, -im);
        *reinterpret_cast<double2*>(Rbig + (size_t)(N + k) * Kp + 2 * b) = make_double2(im, re);
    }
}

// ---- K2a: B = H_m(h_c) . Tx_mat ------------------------------------------------------------------
// slice s of a batch: channel c0 + s / Ms, slice index m = s % Ms.  sum_isi (MATLAB semantics,
// main_interference_calculation.m:198): Ms = 2 and slice 1 holds sum_{m>=1} H_m.
// Bbig[s][kk][j], kk = 2b: Re B[b][j], kk = 2b+1: Im B[b][j]; zero from 2 n_rx up to Kp.
// H_m[b][c] = h[m N0 + b - c] (channel.py:49-52) is non-zero only for b < L - 1 + n_tx - m N0: an ISI slice (m >= 1)
// has isi_rows = L - 1 + tail_tx non-zero rows at most, a PREFIX of K in this layout.  Only round_up(2 isi_rows, 64)
// rows of such a slice are written here and read by the contraction kernels (interf_isi_k).
// Each thread forms BB consecutive rows b of one column j from the BB + L - 1 rows of Tx_mat they share.
constexpr int BB = 8;       // fp64 path
constexpr int BBT = 16;     // TF32 path: more rows per thread = fewer re-reads of Tx_mat (it is L2 bandwidth that bounds the kernel)
__host__ __device__ inline int interf_isi_k(int L, int tail_tx, int n_rx, int Kp) {
    const int rows = L - 1 + tail_tx < n_rx ? L - 1 + tail_tx : n_rx;
    const int k = rows > 0 ? ((2 * rows + 63) / 64) * 64 : 64;   // never empty: the contraction initialises its accumulators
    return k < Kp ? k : Kp;
}
// TILED: the TF32 path's operand is written directly (hi/lo split, UMMA tiles, float4 per 4 consecutive kk); Bbig is
// then the float work buffer and the fp64 B matrix never exists.  That path is fp32-grade by contract (3xTF32), so
// its band product runs in packed FP32 (taps and Tx_mat rounded to fp32, fp32 accumulation: ~1e-7 relative, far
// inside the stated bound) instead of FP64 FMAs, which bound the fp64 variant of this kernel.
// T: Tx_mat as double2 (fp64 path) or float2 (TILED: rounded once by tile_tx_f32, half the bytes per re-read)
template <bool TILED>
__global__ void __launch_bounds__(256) build_b(double* __restrict__ Bbig, const void* __restrict__ Tv,
                                               const double2* __restrict__ chan, int L, int N, int n_tx, int n_rx,
                                               int N0, int Kp, int Ms, int M, int c0, int sum_isi, int k_isi) {
    constexpr int BB = TILED ? BBT : wofdm::BB;
    // taps of this slice's channel in shared memory, zero-padded by BB on both sides: the inner loop needs no
    // range checks and reads them as broadcasts
    extern __shared__ __align__(16) double2 hs_raw[];
    const int s = blockIdx.z, b0 = blockIdx.y * BB;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = c0 + s / Ms, ms = s % Ms;
    const int k_rows = ms == 0 ? Kp : k_isi;                 // rows of this slice that exist for the contraction
    if (2 * b0 >= k_rows) return;                            // (uniform per block)
    using A2 = typename std::conditional<TILED, float2, double2>::type;    // accumulation type
    A2* const hs = reinterpret_cast<A2*>(hs_raw);
    for (int l = threadIdx.x; l < L + 2 * BB; l += blockDim.x) {
        const double2 t = (l >= BB && l < L + BB) ? chan[(size_t)c * L + l - BB] : make_double2(0.0, 0.0);
        hs[l].x = t.x; hs[l].y = t.y;
    }
    __syncthreads();
    if (j >= N) return;
    const A2* h = hs + BB;                                   // h[-BB .. L+BB)
    A2 acc[BB];
#pragma unroll
    for (int i = 0; i < BB; ++i) { acc[i].x = 0; acc[i].y = 0; }
    const int m_lo = ms, m_hi = (sum_isi && ms == 1) ? M - 1 : ms;
    if (b0 < n_rx) {
        for (int m = m_lo; m <= m_hi; ++m) {
            // rows m N0 + b0 - (L-1) .. m N0 + b0 + BB - 1 of Tx_mat: row r feeds output i through tap l = m N0 + b0 + i - r
            const int r_lo = m * N0 + b0 - (L - 1);
            for (int rr = 0; rr < BB + L - 1; ++rr) {
                const int row = r_lo + rr;
                if (row < 0 || row >= n_tx) continue;
                const A2 x = reinterpret_cast<const A2*>(Tv)[(size_t)row * N + j];
                const A2* hw = h + (L - 1) - rr;              // tap of output i: hw[i] (zero outside [0, L))
#pragma unroll
                for (int i = 0; i < BB; ++i) cmac(acc[i], hw[i], x);
            }
        }
    }
    if constexpr (TILED) {
        static_assert(BB % 2 == 0, "two rows b = four consecutive kk = one 16-byte chunk");
        float* bt = reinterpret_cast<float*>(Bbig);
        const int nk = Kp / TF32_KB;
#pragma unroll
        for (int i = 0; i < BB; i += 2) {
            const int kk = 2 * (b0 + i);
            if (kk >= k_rows) break;
            float4 hi, lo;
            tf32_split(b0 + i < n_rx ? acc[i].x : 0.0, hi.x, lo.x);
            tf32_split(b0 + i < n_rx ? acc[i].y : 0.0, hi.y, lo.y);
            tf32_split(b0 + i + 1 < n_rx ? acc[i + 1].x : 0.0, hi.z, lo.z);
            tf32_split(b0 + i + 1 < n_rx ? acc[i + 1].y : 0.0, hi.w, lo.w);
            float* dst = bt + tf32_b_offset(s, nk, N, j, kk);
            *reinterpret_cast<float4*>(dst) = hi;
            *reinterpret_cast<float4*>(dst + (size_t)TF32_TN * TF32_KB) = lo;
        }
    } else {
        double* out = Bbig + (size_t)s * Kp * N;
#pragma unroll
        for (int i = 0; i < BB; ++i) {
            const int b = b0 + i;
            if (2 * b >= k_rows) break;
            const bool live = b < n_rx;
            out[(size_t)(2 * b) * N + j] = live ? acc[i].x : 0.0;
            out[(size_t)(2 * b + 1) * N + j] = live ? acc[i].y : 0.0;
        }
    }
}

// ---- K2b: FP64 tensor-core contraction with fused power epilogue ----------------------------------
constexpr int BM = 128, BN = 64, BK = 16, AS = BK + 4, BS = BN + 4;

__device__ __forceinline__ void dmma8x8x4(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// grid (N / BN column tiles of a slice, 2N / BM row tiles, slices); P[c][k] += row power.
// STORE (window Hessian, K5): no power epilogue, [Re A; Im A] of slice s is written to P + s*2N*N instead.
template <bool STORE>
__global__ void __launch_bounds__(256) gemm_power_f64(const double* __restrict__ Rbig, const double* __restrict__ Bbig,
                                                      double* __restrict__ P, int N, int Kp, int Ms, int c0, int scalar,
                                                      int k_isi) {
    extern __shared__ __align__(16) double gsm[];
    double (*As)[BM * AS] = reinterpret_cast<double (*)[BM * AS]>(gsm);
    double (*Bs)[BK * BS] = reinterpret_cast<double (*)[BK * BS]>(gsm + 2 * BM * AS);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp >> 1) * 32, wn = (warp & 1) * 32;
    const int row0 = blockIdx.y * BM, col0 = blockIdx.x * BN, s = blockIdx.z;
    const double* A = Rbig + (size_t)row0 * Kp;
    const double* B = Bbig + (size_t)s * Kp * N + col0;
    const int ar = tid >> 1, ak = (tid & 1) * 8;          // A tile: 128 rows x 16, 8 doubles per thread
    const int br = tid >> 4, bc = (tid & 15) * 4;         // B tile: 16 rows x 64, 4 doubles per thread
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jn = 0; jn < 4; ++jn) acc[i][jn][0] = acc[i][jn][1] = 0.0;
    double ra[8], rb[4];
    auto gload = [&](int k0) {
        const double4* pa = reinterpret_cast<const double4*>(A + (size_t)ar * Kp + k0 + ak);
        const double4 a0 = pa[0], a1 = pa[1];
        ra[0] = a0.x; ra[1] = a0.y; ra[2] = a0.z; ra[3] = a0.w; ra[4] = a1.x; ra[5] = a1.y; ra[6] = a1.z; ra[7] = a1.w;
        const double4 b0 = *reinterpret_cast<const double4*>(B + (size_t)(k0 + br) * N + bc);
        rb[0] = b0.x; rb[1] = b0.y; rb[2] = b0.z; rb[3] = b0.w;
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int i = 0; i < 8; ++i) As[buf][ar * AS + ak + i] = ra[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) Bs[buf][br * BS + bc + i] = rb[i];
    };
    gload(0);
    sstore(0);
    __syncthreads();
    const int nk = ((s % Ms) == 0 ? Kp : k_isi) / BK;        // ISI slices: only their non-zero K prefix (build_b)
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * BK);
#pragma unroll
        for (int kk = 0; kk < BK; kk += 4) {
            double fa[4], fb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) fa[i] = As[buf][(wm + 8 * i + (lane >> 2)) * AS + kk + (lane & 3)];
#pragma unroll
            for (int jn = 0; jn < 4; ++jn) fb[jn] = Bs[buf][(kk + (lane & 3)) * BS + wn + 8 * jn + (lane >> 2)];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) dmma8x8x4(acc[i][jn][0], acc[i][jn][1], fa[i], fb[jn]);
        }
        if (kt + 1 < nk) sstore(buf ^ 1);
        __syncthreads();
    }
    if constexpr (STORE) {
        double* out = P + (size_t)s * 2 * N * N;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = row0 + wm + 8 * i + (lane >> 2);
#pragma unroll
            for (int jn = 0; jn < 4; ++jn) {
                const int jcol = col0 + wn + 8 * jn + 2 * (lane & 3);
                *reinterpret_cast<double2*>(out + (size_t)r * N + jcol) = make_double2(acc[i][jn][0], acc[i][jn][1]);
            }
        }
        return;
    }
    // epilogue: rows r (Re) and N + r (Im) of big-A both belong to sub-carrier r; slice 0 drops j == k
    const int c = c0 + s / Ms, ms = s % Ms;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = row0 + wm + 8 * i + (lane >> 2);
        const int k = r % N;
        double pw = 0.0;
#pragma unroll
        for (int jn = 0; jn < 4; ++jn)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int jcol = col0 + wn + 8 * jn + 2 * (lane & 3) + e;
                const double v = acc[i][jn][e];
                if (!(ms == 0 && jcol == k)) pw = fma(v, v, pw);
            }
        pw += __shfl_xor_sync(0xffffffffu, pw, 1);
        pw += __shfl_xor_sync(0xffffffffu, pw, 2);
        if ((lane & 3) == 0) atomicAdd(scalar ? &P[c] : &P[(size_t)c * N + k], pw);
    }
}

int interf_upload(wofdm_ctx* h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                  const double* chan, int L, int C, int mode, InterfDev* out) {
    DeviceCtx& d = h->devs[0];
    const int N = sys->N, n_tx = N + sys->cp + sys->cs, n_rx = n_tx - sys->tail_tx;
    InterfDev v;
    v.N = N; v.n_tx = n_tx; v.n_rx = n_rx; v.N0 = n_rx;
    v.Kp = ((2 * n_rx + 63) / 64) * 64;
    v.M = 1 + (L - 1 + sys->tail_tx + n_rx - 1) / n_rx;     // channel.py:42
    const size_t bytes = (size_t)(n_tx + N + sys->tail_rx) * 8 + (size_t)L * C * 16 + (size_t)n_tx * N * 16 +
                         (size_t)2 * N * v.Kp * 8;
    // batch of channels whose B matrices fit the staging budget (1 GiB of the arena).  Measured and not kept: batches small
    // enough for the staging buffer to stay inside the 126 MB L2 (so that the operand never travels to HBM and back: one
    // 250-channel call moves 331 MB) -- 1.70 -> 2.31 ms (fp64) and 0.43 -> 0.74 ms (TF32) at 48 MB: the call is bound by its
    // kernels, not by that traffic, and short batches quantise badly over 148 SMs (DESIGN.md section 4).
    const size_t per_chan = (size_t)v.M * v.Kp * N * 8;
    const size_t budget = (size_t)1 << 30;
    v.batch = (int)std::max<size_t>(1, std::min<size_t>((size_t)C, budget / per_chan));
    const size_t tf32_bytes = mode == 1 ? ((size_t)2 * 2 * N * v.Kp + (size_t)2 * v.batch * v.M * N * v.Kp) * 4 : 0;
    const size_t t32_bytes = mode == 1 ? (size_t)n_tx * N * 8 : 0;
    int rc = arena_reserve(h, d, bytes + (size_t)v.batch * per_chan + (size_t)C * N * 8 + tf32_bytes + t32_bytes + 256);
    if (rc) return rc;
    v.vtx = static_cast<double*>(arena_take(d, (size_t)n_tx * 8));
    v.vrx = static_cast<double*>(arena_take(d, (size_t)(N + sys->tail_rx) * 8));
    v.chan = static_cast<double2*>(arena_take(d, (size_t)L * C * 16));
    v.T = static_cast<double2*>(arena_take(d, (size_t)n_tx * N * 16));
    v.Rbig = static_cast<double*>(arena_take(d, (size_t)2 * N * v.Kp * 8));
    v.Bbig = static_cast<double*>(arena_take(d, (size_t)v.batch * per_chan));
    v.P = static_cast<double*>(arena_take(d, (size_t)C * N * 8));
    v.tf32_work = tf32_bytes ? static_cast<float*>(arena_take(d, tf32_bytes)) : nullptr;
    v.T32 = t32_bytes ? static_cast<float2*>(arena_take(d, t32_bytes)) : nullptr;
    if (t32_bytes && !v.T32) return fail(h, WOFDM_ENOMEM, "arena exhausted");
    if ((tf32_bytes && !v.tf32_work) || !v.vtx || !v.vrx || !v.chan || !v.T || !v.Rbig || !v.Bbig || !v.P) return fail(h, WOFDM_ENOMEM, "arena exhausted");
    WOFDM_CUDA(h, cudaMemcpyAsync(v.vtx, win_tx, (size_t)n_tx * 8, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(v.vrx, win_rx, (size_t)(N + sys->tail_rx) * 8, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(v.chan, chan, (size_t)L * C * 16, cudaMemcpyHostToDevice, d.stream));
    build_tx_matrix<<<n_tx, 256, 0, d.stream>>>(v.T, v.vtx, N, sys->cp, n_tx, v.T32);
    build_rx_matrix<<<N, 256, 0, d.stream>>>(v.Rbig, v.vrx, N, sys->tail_rx, sys->rm, sys->shift, n_rx, v.Kp);
    WOFDM_CUDA(h, cudaGetLastError());
    h->launches += 2;
    *out = v;
    return WOFDM_OK;
}

static int interf_run_quad(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                           const double* chan, int L, int C, int scalar, double* P);

static int interf_run(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                      const double* chan, int L, int C, int mode, int scalar, double* P) {
    NvtxRange nvtx_("wofdm_interf_power");
    if (!h) return WOFDM_EINVAL;
    int rc = validate_sys(h, sys, L);
    if (rc) return rc;
    if (!win_tx || !win_rx || !chan || !P || C < 1) return fail(h, WOFDM_EINVAL, "bad buffer");
    if (mode != 0 && mode != 1 && mode != 2) return fail(h, WOFDM_EINVAL, "mode must be 0 (fp64), 1 (TF32-split) or 2 (fp64, Hermitian form in the taps)");
    if (sys->N % 64) return fail(h, WOFDM_EUNSUPPORTED, "interference path needs N to be a multiple of 64");
    if (mode == 2) return interf_run_quad(h, sys, win_tx, win_rx, chan, L, C, scalar, P);
    if (mode == 1 && sys->N % TF32_TN) return fail(h, WOFDM_EUNSUPPORTED, "TF32-split interference path needs N to be a multiple of 256");
    DeviceCtx& d = h->devs[0];
    WOFDM_CUDA(h, cudaSetDevice(d.dev));
    for (auto& e : h->interf_ev)
        if (!e) WOFDM_CUDA(h, cudaEventCreate(&e));
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[0], d.stream));
    InterfDev v;
    rc = interf_upload(h, sys, win_tx, win_rx, chan, L, C, mode, &v);
    if (rc) return rc;
    const bool one_batch = v.batch >= C;             // (the kernel times are taken for single-batch calls)
    const int N = sys->N;
    const size_t pbytes = scalar ? (size_t)C * 8 : (size_t)C * N * 8;
    WOFDM_CUDA(h, cudaMemsetAsync(v.P, 0, pbytes, d.stream));
    const int Ms = scalar ? std::min(v.M, 2) : v.M;      // scalar: slice 1 = sum of the ISI slices
    const int k_isi = interf_isi_k(L, sys->tail_tx, v.n_rx, v.Kp);
    for (int c0 = 0; c0 < C; c0 += v.batch) {
        const int nc = std::min(v.batch, C - c0);
        const int slices = nc * Ms;
        const bool tiled = mode == 1;                         // the TF32 operand straight from the band product
        const int bb = tiled ? BBT : BB;
        if (one_batch) WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[1], d.stream));
        const dim3 bgrid((N + 255) / 256, (v.Kp / 2 + bb - 1) / bb, slices);
        const size_t bsm = (size_t)(L + 2 * bb) * sizeof(double2);
        if (tiled)
            build_b<true><<<bgrid, 256, bsm, d.stream>>>(reinterpret_cast<double*>(interf_tf32_b_tiles(v, N)), v.T32, v.chan, L, N,
                                                        v.n_tx, v.n_rx, v.N0, v.Kp, Ms, v.M, c0, scalar, k_isi);
        else
            build_b<false><<<bgrid, 256, bsm, d.stream>>>(v.Bbig, v.T, v.chan, L, N, v.n_tx, v.n_rx, v.N0, v.Kp, Ms, v.M, c0,
                                                         scalar, k_isi);
        WOFDM_CUDA(h, cudaGetLastError());
        if (one_batch) WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[2], d.stream));
        if (mode == 0) {
            constexpr size_t smem = (size_t)(2 * BM * AS + 2 * BK * BS) * sizeof(double);
            WOFDM_CUDA(h, cudaFuncSetAttribute(gemm_power_f64<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            gemm_power_f64<false><<<dim3(N / BN, 2 * N / BM, slices), 256, smem, d.stream>>>(v.Rbig, v.Bbig, v.P, N, v.Kp, Ms, c0, scalar, k_isi);
            WOFDM_CUDA(h, cudaGetLastError());
        } else {
            rc = interf_gemm_tf32(h, sys, v, Ms, c0, slices, scalar, k_isi);
            if (rc) return rc;
        }
        if (one_batch) WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[3], d.stream));
        h->launches += 2;
    }
    WOFDM_CUDA(h, cudaMemcpyAsync(P, v.P, pbytes, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[4], d.stream));
    WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
    float ms = 0.f;
    h->interf_ms[0] = h->interf_ms[1] = h->interf_ms[2] = -1.0;
    if (cudaEventElapsedTime(&ms, h->interf_ev[0], h->interf_ev[4]) == cudaSuccess) h->interf_ms[0] = ms;
    if (one_batch) {
        if (cudaEventElapsedTime(&ms, h->interf_ev[1], h->interf_ev[2]) == cudaSuccess) h->interf_ms[1] = ms;
        if (cudaEventElapsedTime(&ms, h->interf_ev[2], h->interf_ev[3]) == cudaSuccess) h->interf_ms[2] = ms;
    }
    h->interf_k_isi = k_isi; h->interf_kp = v.Kp;
    return WOFDM_OK;
}

// ---- K2 mode 2: the interference power as a Hermitian form in the channel taps ---------------------------------------
// H_m(h) is linear in the taps, so A_m(c) = sum_l h_c[l] G_{m,l} with G_{m,l} = Rx_mat . H_m(e_l) . Tx_mat the response to
// the unit impulse at tap l, and
//     P_k(c) = sum_{l,l'} h_c[l] conj(h_c[l']) Q_k[l,l'],   Q_k[l,l'] = sum_m sum_{j (!= k for m = 0)} G_{m,l}[k,j] conj(G_{m,l'}[k,j]).
// The window pair costs L impulse responses through the SAME band product and tensor-core contraction as mode 0 (store
// epilogue) plus N small Gram matrices; every channel realisation then costs L^2 complex MACs per sub-carrier instead of a
// 2N x K x N GEMM per slice, and nothing per channel travels through HBM but its taps and its row of P.  Same
// arithmetic type (fp64), same off-diagonal mask before squaring, so no cancellation the direct form does not have.
// (interf_calc.py:91-100 evaluates ONE channel per call; the 250-channel sweeps of BASELINE configs[3] / the 10 000
// channels of configs[4] are where this pays: the cost no longer grows with the number of channels.)
// In real arithmetic (Q_k is Hermitian): P_k(c) = w_c . q_k over F = L (L + 1) features, two per tap pair p = (l, l' <= l):
//   q_k[2p] = Re Q_k[l,l'], q_k[2p+1] = Im Q_k[l,l'];   w_c[2p] = 2 Re(h_l conj h_l'), w_c[2p+1] = -2 Im(h_l conj h_l')
//   (l = l': |h_l|^2 and 0), so all channels and sub-carriers are ONE real product P = W . Q^T  (C x F x N).
__host__ __device__ inline int quad_features(int L) { return ((L * (L + 1) + 15) / 16) * 16; }   // padded to the K tile
__device__ __forceinline__ void quad_pair(int p, int& l, int& lp) {
    l = (int)((sqrt(8.0 * p + 1.0) - 1.0) * 0.5);
    while ((l + 1) * (l + 2) / 2 <= p) ++l;
    while (l * (l + 1) / 2 > p) --l;
    lp = p - l * (l + 1) / 2;
}
// One CTA per sub-carrier k; X[l*Ms + ms] = [Re G; Im G] (2N x N) from gemm_power_f64<true>.  qf: [N][F].
// Q_k = Z Z^H with Z[l][(ms, j)] the k-th rows of the impulse responses (the diagonal entry of slice 0 masked): a thread
// owns a 4 x 4 block of tap pairs (32 fp64 accumulators: 16 shared-memory loads per 64 FMAs) and every G-th column of the
// staged tile; the G column groups of a block meet in shared memory at the end.
template <int JT>
__global__ void __launch_bounds__(256) quad_q_kernel(const double* __restrict__ X, double* __restrict__ qf, int N, int L, int Ms, int F) {
    extern __shared__ __align__(16) double qsm[];            // [LB4*4*Ms*2][JT + 1] (odd pitch), then the block sums [nblk][32]
    constexpr int JP = JT + 1;
    const int k = blockIdx.x;
    const size_t mat = (size_t)2 * N * N;
    const int LB4 = (L + 3) / 4, nblk = LB4 * (LB4 + 1) / 2, LP = 4 * LB4;
    int G = 1;
    while (2 * G * nblk <= 256 && 2 * G <= 8) G *= 2;        // column groups per block: 1, 2, 4 or 8
    double* const qsum = qsm + (size_t)LP * Ms * 2 * JP;
    const int blk = threadIdx.x / G, grp = threadIdx.x % G;
    const bool live = blk < nblk;
    int br = 0, bc = 0;                                       // block row >= block column
    if (live) quad_pair(blk, br, bc);
    double ar[4][4], ai[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) ar[i][j] = ai[i][j] = 0.0;
    for (int j0 = 0; j0 < N; j0 += JT) {
        __syncthreads();
        constexpr int UL = 6;                                 // loads in flight per thread (the tile is L2 / HBM latency bound)
        for (int e0 = threadIdx.x; e0 < LP * Ms * 2 * JT; e0 += 256 * UL) {
            double v[UL];
#pragma unroll
            for (int u = 0; u < UL; ++u) {
                const int e = e0 + 256 * u, j = e % JT, row = e / JT, part = row & 1, sl = row >> 1;   // sl = l * Ms + ms
                v[u] = 0.0;
                if (sl < L * Ms) v[u] = __ldg(X + (size_t)sl * mat + (size_t)(part * N + k) * N + j0 + j);
            }
#pragma unroll
            for (int u = 0; u < UL; ++u) {
                const int e = e0 + 256 * u, j = e % JT, row = e / JT, sl = row >> 1;
                if (e < LP * Ms * 2 * JT) qsm[row * JP + j] = (sl % Ms == 0 && j0 + j == k) ? 0.0 : v[u];   // slice 0: off-diagonal entries only
            }
        }
        __syncthreads();
        if (live) {
            for (int ms = 0; ms < Ms; ++ms) {
                const double* xb = qsm + (size_t)((4 * br * Ms + ms) * 2) * JP;       // row l = 4 br + i: xb + i * Ms * 2 * JP (re), + JP (im)
                const double* yb = qsm + (size_t)((4 * bc * Ms + ms) * 2) * JP;
                for (int j = grp; j < JT; j += G) {
                    double xr[4], xi[4], yr[4], yi[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        xr[i] = xb[(size_t)i * Ms * 2 * JP + j]; xi[i] = xb[(size_t)i * Ms * 2 * JP + JP + j];
                        yr[i] = yb[(size_t)i * Ms * 2 * JP + j]; yi[i] = yb[(size_t)i * Ms * 2 * JP + JP + j];
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int jj = 0; jj < 4; ++jj) {     // G_l conj(G_l')
                            ar[i][jj] = fma(xr[i], yr[jj], fma(xi[i], yi[jj], ar[i][jj]));
                            ai[i][jj] = fma(xi[i], yr[jj], fma(-xr[i], yi[jj], ai[i][jj]));
                        }
                }
            }
        }
    }
    // the G column groups of a block are G consecutive lanes: butterfly sum, then group 0 publishes the block
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
            for (int st = 1; st < G; st <<= 1) {
                ar[i][jj] += __shfl_xor_sync(0xffffffffu, ar[i][jj], st);
                ai[i][jj] += __shfl_xor_sync(0xffffffffu, ai[i][jj], st);
            }
            if (live && grp == 0) {
                qsum[blk * 32 + (i * 4 + jj) * 2] = ar[i][jj];
                qsum[blk * 32 + (i * 4 + jj) * 2 + 1] = ai[i][jj];
            }
        }
    __syncthreads();
    for (int e = threadIdx.x; e < nblk * 16; e += 256) {
        int r, c;
        quad_pair(e / 16, r, c);
        const int l = 4 * r + (e % 16) / 4, lp = 4 * c + (e % 4);
        if (l < L && lp <= l)
            *reinterpret_cast<double2*>(qf + (size_t)k * F + 2 * (l * (l + 1) / 2 + lp)) = make_double2(qsum[2 * e], qsum[2 * e + 1]);
    }
    for (int f = L * (L + 1) + threadIdx.x; f < F; f += 256) qf[(size_t)k * F + f] = 0.0;
}

// wf: [C][F], the channels' tap-pair features
__global__ void __launch_bounds__(256) quad_w_kernel(const double2* __restrict__ chan, double* __restrict__ wf, int L, int C, int F) {
    const int c = blockIdx.y, npair = L * (L + 1) / 2;
    const double2* h = chan + (size_t)c * L;
    for (int p = blockIdx.x * 256 + threadIdx.x; 2 * p < F; p += gridDim.x * 256) {
        double2 w = make_double2(0.0, 0.0);
        if (p < npair) {
            int l, lp;
            quad_pair(p, l, lp);
            const double2 a = h[l], b = h[lp];
            if (l == lp) w.x = a.x * a.x + a.y * a.y;
            else { w.x = 2.0 * (a.x * b.x + a.y * b.y); w.y = -2.0 * (a.y * b.x - a.x * b.y); }
        }
        *reinterpret_cast<double2*>(wf + (size_t)c * F + 2 * p) = w;
    }
}

// P[c][k] = sum_f wf[c][f] qf[k][f]: a TS x TS tile per CTA (64, or 32 when 64 would leave most SMs idle), RT x RT outputs
// per thread, F in tiles of 16 (plain FP64 FMAs: the product is C x L(L+1) x N, 0.06 GFLOP for the 250 channels of
// configs[3]).  scalar: the row sum over k instead.
// (also the Gram product of the window Hessian's parts: ldw / ldq = row pitches, F = features contracted, scale on the way out;
// ACC: P += scale * product instead of P = ..., for the channel-set Hessian's passes after the first -- non-scalar only)
template <int TS, bool ACC = false>
__global__ void __launch_bounds__(256) quad_eval_kernel(const double* __restrict__ wf, const double* __restrict__ qf,
                                                        double* __restrict__ P, int N, int C, int F, int scalar,
                                                        size_t ldw, size_t ldq, double scale) {
    constexpr int RT = TS / 16;
    __shared__ double ws[16][TS + 4], qs[16][TS + 4];
    const int c0 = blockIdx.x * TS, k0 = blockIdx.y * TS;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // outputs: channels c0 + RT ty + i, sub-carriers k0 + RT tx + j
    // loads: TS rows x 16 features per operand = TS * 16 / 256 doubles per thread
    constexpr int LV = TS / 16;                                      // consecutive features per thread (4 or 2)
    const int lr = threadIdx.x / (16 / LV), lf = (threadIdx.x % (16 / LV)) * LV;
    double acc[RT][RT];
#pragma unroll
    for (int i = 0; i < RT; ++i)
#pragma unroll
        for (int j = 0; j < RT; ++j) acc[i][j] = 0.0;
    for (int f0 = 0; f0 < F; f0 += 16) {
        double a[LV], b[LV];
#pragma unroll
        for (int i = 0; i < LV; ++i) {
            a[i] = c0 + lr < C ? wf[(size_t)(c0 + lr) * ldw + f0 + lf + i] : 0.0;
            b[i] = k0 + lr < N ? qf[(size_t)(k0 + lr) * ldq + f0 + lf + i] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < LV; ++i) { ws[lf + i][lr] = a[i]; qs[lf + i][lr] = b[i]; }
        __syncthreads();
#pragma unroll
        for (int f = 0; f < 16; ++f) {
            double wv[RT], qv[RT];
#pragma unroll
            for (int i = 0; i < RT; ++i) { wv[i] = ws[f][RT * ty + i]; qv[i] = qs[f][RT * tx + i]; }
#pragma unroll
            for (int i = 0; i < RT; ++i)
#pragma unroll
                for (int j = 0; j < RT; ++j) acc[i][j] = fma(wv[i], qv[j], acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < RT; ++i) {
        const int c = c0 + RT * ty + i;
        if (c >= C) continue;
        if (scalar) {
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < RT; ++j) if (k0 + RT * tx + j < N) sum += acc[i][j];
            atomicAdd(&P[c], scale * sum);
        } else {
#pragma unroll
            for (int j = 0; j < RT; ++j) {
                if (k0 + RT * tx + j >= N) continue;
                double* const o = P + (size_t)c * N + k0 + RT * tx + j;
                *o = ACC ? *o + scale * acc[i][j] : scale * acc[i][j];
            }
        }
    }
}

static int interf_run_quad(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                           const double* chan, int L, int C, int scalar, double* P) {
    DeviceCtx& d = h->devs[0];
    WOFDM_CUDA(h, cudaSetDevice(d.dev));
    for (auto& e : h->interf_ev)
        if (!e) WOFDM_CUDA(h, cudaEventCreate(&e));
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[0], d.stream));
    static cudaEvent_t dbg[4] = {nullptr, nullptr, nullptr, nullptr};
    const bool dbg_on = getenv("WOFDM_DEBUG") != nullptr;
    if (dbg_on) for (auto& e : dbg) if (!e) cudaEventCreate(&e);
    const int N = sys->N, n_tx = N + sys->cp + sys->cs, n_rx = n_tx - sys->tail_tx, n_w = N + sys->tail_rx;
    const int Kp = ((2 * n_rx + 63) / 64) * 64;
    const int M = 1 + (L - 1 + sys->tail_tx + n_rx - 1) / n_rx;
    const int Ms = scalar ? std::min(M, 2) : M;
    const int k_isi = interf_isi_k(L, sys->tail_tx, n_rx, Kp);
    if (L > 88) return fail(h, WOFDM_EUNSUPPORTED, "mode 2: at most 88 taps (253 blocks of 4 x 4 tap pairs per CTA)");
    const size_t mat = (size_t)2 * N * N * 8;
    const int F = quad_features(L);
    const size_t pbytes = scalar ? (size_t)C * 8 : (size_t)C * N * 8;
    const size_t need = (size_t)(n_tx + n_w) * 8 + (size_t)L * C * 16 + (size_t)L * L * 16 + (size_t)n_tx * N * 16 +
                        (size_t)2 * N * Kp * 8 + (size_t)L * Ms * Kp * N * 8 + (size_t)L * Ms * mat + (size_t)(N + C) * F * 8 + pbytes + 4096;
    int rc = arena_reserve(h, d, need);
    if (rc) return rc;
    double* d_vtx = static_cast<double*>(arena_take(d, (size_t)n_tx * 8));
    double* d_vrx = static_cast<double*>(arena_take(d, (size_t)n_w * 8));
    double2* d_chan = static_cast<double2*>(arena_take(d, (size_t)L * C * 16));
    double2* d_imp = static_cast<double2*>(arena_take(d, (size_t)L * L * 16));
    double2* d_T = static_cast<double2*>(arena_take(d, (size_t)n_tx * N * 16));
    double* d_R = static_cast<double*>(arena_take(d, (size_t)2 * N * Kp * 8));
    double* d_B = static_cast<double*>(arena_take(d, (size_t)L * Ms * Kp * N * 8));
    double* d_X = static_cast<double*>(arena_take(d, (size_t)L * Ms * mat));
    double* d_Q = static_cast<double*>(arena_take(d, (size_t)N * F * 8));
    double* d_W = static_cast<double*>(arena_take(d, (size_t)C * F * 8));
    double* d_P = static_cast<double*>(arena_take(d, pbytes));
    if (!d_vtx || !d_vrx || !d_chan || !d_imp || !d_T || !d_R || !d_B || !d_X || !d_Q || !d_W || !d_P) return fail(h, WOFDM_ENOMEM, "arena exhausted");
    std::vector<double> imp((size_t)L * L * 2, 0.0);
    for (int l = 0; l < L; ++l) imp[((size_t)l * L + l) * 2] = 1.0;          // "channel" l = the unit impulse at tap l
    WOFDM_CUDA(h, cudaMemcpyAsync(d_vtx, win_tx, (size_t)n_tx * 8, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(d_vrx, win_rx, (size_t)n_w * 8, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(d_chan, chan, (size_t)L * C * 16, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(d_imp, imp.data(), (size_t)L * L * 16, cudaMemcpyHostToDevice, d.stream));
    build_tx_matrix<<<n_tx, 256, 0, d.stream>>>(d_T, d_vtx, N, sys->cp, n_tx);
    build_rx_matrix<<<N, 256, 0, d.stream>>>(d_R, d_vrx, N, sys->tail_rx, sys->rm, sys->shift, n_rx, Kp);
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[1], d.stream));
    const int slices = L * Ms;
    build_b<false><<<dim3((N + 255) / 256, (Kp / 2 + BB - 1) / BB, slices), 256, (size_t)(L + 2 * BB) * sizeof(double2), d.stream>>>(
        d_B, d_T, d_imp, L, N, n_tx, n_rx, n_rx, Kp, Ms, M, 0, scalar, k_isi);
    WOFDM_CUDA(h, cudaGetLastError());
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[2], d.stream));
    constexpr size_t smem = (size_t)(2 * BM * AS + 2 * BK * BS) * sizeof(double);
    WOFDM_CUDA(h, cudaFuncSetAttribute(gemm_power_f64<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gemm_power_f64<true><<<dim3(N / BN, 2 * N / BM, slices), 256, smem, d.stream>>>(d_R, d_B, d_X, N, Kp, Ms, 0, 0, k_isi);
    WOFDM_CUDA(h, cudaGetLastError());
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[3], d.stream));
    // Gram matrices of the impulse responses and the channels' tap-pair features, then every channel in one product
    const int LB4 = (L + 3) / 4;
    auto q_smem = [&](int jt) { return ((size_t)4 * LB4 * Ms * 2 * (jt + 1) + (size_t)LB4 * (LB4 + 1) / 2 * 32) * sizeof(double); };
    if (q_smem(32) > 220 * 1024) return fail(h, WOFDM_EUNSUPPORTED, "mode 2: the impulse responses of this many taps and slices do not fit shared memory (use mode 0)");
    if (q_smem(64) <= 160 * 1024 && N % 64 == 0) {          // 64 columns per staged tile where they fit (fewer barriers), else 32
        WOFDM_CUDA(h, cudaFuncSetAttribute(quad_q_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)q_smem(64)));
        quad_q_kernel<64><<<N, 256, q_smem(64), d.stream>>>(d_X, d_Q, N, L, Ms, F);
    } else {
        WOFDM_CUDA(h, cudaFuncSetAttribute(quad_q_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)q_smem(32)));
        quad_q_kernel<32><<<N, 256, q_smem(32), d.stream>>>(d_X, d_Q, N, L, Ms, F);
    }
    if (dbg_on) cudaEventRecord(dbg[0], d.stream);
    quad_w_kernel<<<dim3((F / 2 + 255) / 256, C), 256, 0, d.stream>>>(d_chan, d_W, L, C, F);
    if (dbg_on) cudaEventRecord(dbg[1], d.stream);
    WOFDM_CUDA(h, cudaGetLastError());
    if (scalar) WOFDM_CUDA(h, cudaMemsetAsync(d_P, 0, pbytes, d.stream));
    if (((C + 63) / 64) * ((N + 63) / 64) >= 148)
        quad_eval_kernel<64><<<dim3((C + 63) / 64, (N + 63) / 64), 256, 0, d.stream>>>(d_W, d_Q, d_P, N, C, F, scalar, F, F, 1.0);
    else
        quad_eval_kernel<32><<<dim3((C + 31) / 32, (N + 31) / 32), 256, 0, d.stream>>>(d_W, d_Q, d_P, N, C, F, scalar, F, F, 1.0);
    if (dbg_on) cudaEventRecord(dbg[2], d.stream);
    WOFDM_CUDA(h, cudaGetLastError());
    h->launches += 7;
    WOFDM_CUDA(h, cudaMemcpyAsync(P, d_P, pbytes, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaEventRecord(h->interf_ev[4], d.stream));
    WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
    float ms = 0.f;
    h->interf_ms[0] = h->interf_ms[1] = h->interf_ms[2] = -1.0;
    if (cudaEventElapsedTime(&ms, h->interf_ev[0], h->interf_ev[4]) == cudaSuccess) h->interf_ms[0] = ms;
    if (cudaEventElapsedTime(&ms, h->interf_ev[1], h->interf_ev[2]) == cudaSuccess) h->interf_ms[1] = ms;
    if (cudaEventElapsedTime(&ms, h->interf_ev[2], h->interf_ev[3]) == cudaSuccess) h->interf_ms[2] = ms;
    if (dbg_on) {
        float t[6];
        cudaEventElapsedTime(&t[0], h->interf_ev[0], h->interf_ev[1]); cudaEventElapsedTime(&t[1], h->interf_ev[3], dbg[0]);
        cudaEventElapsedTime(&t[2], dbg[0], dbg[1]); cudaEventElapsedTime(&t[3], dbg[1], dbg[2]); cudaEventElapsedTime(&t[4], dbg[2], h->interf_ev[4]);
        fprintf(stderr, "[wofdm] mode 2: upload+builders %.3f, Q %.3f, W %.3f, eval %.3f, download %.3f ms\n", t[0], t[1], t[2], t[3], t[4]);
    }
    h->interf_k_isi = k_isi; h->interf_kp = Kp;
    return WOFDM_OK;
}

// ---- K5: window-optimisation Hessian (SURVEY.md section 8f-2) ----------------------------------------
// H[u,u'] = 2 Re( <offdiag A0_u, offdiag A0_u'> + <AS_u, AS_u'> ), A0_u / AS_u = the K2 contraction for the basis window
// pair u = (Rx basis a, Tx basis b) on slice 0 / on the sum of the ISI slices.  Replaces the O(n^2 N^2) loops of
// OptimizerTx/Rx/TxRx.gen_hessian (python/optimization_tools/optimizers.py:132-175, 232-257, 427-507, 808-833) and
// quad_objective_tx/_rx (matlab/window_optimization.m:596-680).  X[u][ms][2N][N] holds [Re A; Im A].
// ACC: H += the Gram entries (passes after the first of a channel set); otherwise H = them, so that whatever H held before
// never enters the sum.
template <bool ACC>
__global__ void __launch_bounds__(256) gram_offdiag(const double* __restrict__ X, double* __restrict__ H, int n_var, int N,
                                                    int n_tb) {
    __shared__ double red[256];
    // pair index -> (u, u'), u' <= u
    int u = 0, rem = blockIdx.x;
    while (rem > u) { rem -= u + 1; ++u; }
    const int up = rem;
    const size_t mat = (size_t)2 * N * N;                    // one [Re A; Im A]
    // X layout: [a][b][ms][2N][N] with u = a*n_tb + b
    const double* x0 = X + (size_t)u * 2 * mat;
    const double* y0 = X + (size_t)up * 2 * mat;
    double acc = 0.0;
    for (size_t e = threadIdx.x; e < 2 * mat; e += 256) {
        const int ms = (int)(e / mat);
        const size_t w = e - (size_t)ms * mat;
        const int r = (int)(w / N), j = (int)(w - (size_t)r * N);
        if (ms == 0 && j == r % N) continue;                  // slice 0: off-diagonal entries only
        acc = fma(x0[e], y0[e], acc);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
        if (threadIdx.x < st) red[threadIdx.x] += red[threadIdx.x + st];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double g = 2.0 * red[0];
        if (ACC) {
            H[(size_t)u * n_var + up] += g;
            if (up != u) H[(size_t)up * n_var + u] += g;          // (a diagonal entry is one element: add once)
        } else {
            H[(size_t)u * n_var + up] = g;
            H[(size_t)up * n_var + u] = g;
        }
    }
    (void)n_tb;
}

// slice 0 of every stored [Re A; Im A]: the diagonal entries leave the sums (off-diagonal interference only)
__global__ void zero_diag_kernel(double* __restrict__ X, int n_var, int N) {
    const int u = blockIdx.x;
    double* x = X + (size_t)u * 2 * ((size_t)2 * N * N);
    for (int k = threadIdx.x; k < N; k += blockDim.x) { x[(size_t)k * N + k] = 0.0; x[(size_t)(N + k) * N + k] = 0.0; }
}

// bt: n_tb Tx windows (n_tx each), br: n_rb Rx windows (N + tail_rx each), host.  H_out (sum of the parts, gram_offdiag) or
// the parts H_ici / H_isi (Gram products through quad_eval_kernel); n_var = n_rb * n_tb, u = a * n_tb + b.
// chan: r impulse responses of L taps back to back; the result is the SUM over them of each one's Hessian: one pass of the
// band product and the contraction per response, the first pass storing the Gram products and every later one adding to
// them on the device.  The basis operands Tx_mat(t_b) / Rbig(r_a) do not depend on the channel and are built once.
static int window_hessian_core(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, int r, const double* bt_h,
                               int n_tb, const double* br_h, int n_rb, double* H_out, double* H_ici, double* H_isi) {
    DeviceCtx& d = h->devs[0];
    WOFDM_CUDA(h, cudaSetDevice(d.dev));
    for (auto& e : h->hess_ev)
        if (!e) WOFDM_CUDA(h, cudaEventCreate(&e));
    WOFDM_CUDA(h, cudaEventRecord(h->hess_ev[0], d.stream));
    const int N = sys->N, n_tx = N + sys->cp + sys->cs, n_rx = n_tx - sys->tail_tx, n_w = N + sys->tail_rx;
    const int n_var = n_tb * n_rb;
    const int Kp = ((2 * n_rx + 63) / 64) * 64;
    const int M = 1 + (L - 1 + sys->tail_tx + n_rx - 1) / n_rx;
    const int Ms = 2;                                          // slice 0 and the sum of the ISI slices
    const int k_isi = interf_isi_k(L, sys->tail_tx, n_rx, Kp);
    const size_t matb = (size_t)2 * N * N * 8;
    const size_t t_one = (size_t)n_tx * N, r_one = (size_t)2 * N * Kp;     // elements of one Tx_mat (double2) / one Rbig
    const size_t need = (size_t)n_tb * n_tx * 8 + (size_t)n_rb * n_w * 8 + (size_t)r * L * 16 + (size_t)n_tb * t_one * 16 +
                        (size_t)n_rb * r_one * 8 + (size_t)n_tb * Ms * Kp * N * 8 + (size_t)n_var * Ms * matb + (size_t)2 * n_var * n_var * 8;
    int rc = arena_reserve(h, d, need);
    if (rc) return rc;
    double* d_bt = static_cast<double*>(arena_take(d, (size_t)n_tb * n_tx * 8));
    double* d_br = static_cast<double*>(arena_take(d, (size_t)n_rb * n_w * 8));
    double2* d_chan = static_cast<double2*>(arena_take(d, (size_t)r * L * 16));
    double2* d_T = static_cast<double2*>(arena_take(d, (size_t)n_tb * t_one * 16));
    double* d_R = static_cast<double*>(arena_take(d, (size_t)n_rb * r_one * 8));
    double* d_B = static_cast<double*>(arena_take(d, (size_t)n_tb * Ms * Kp * N * 8));
    double* d_X = static_cast<double*>(arena_take(d, (size_t)n_var * Ms * matb));
    double* d_H = static_cast<double*>(arena_take(d, (size_t)2 * n_var * n_var * 8));
    if (!d_bt || !d_br || !d_chan || !d_T || !d_R || !d_B || !d_X || !d_H) return fail(h, WOFDM_ENOMEM, "arena exhausted");
    WOFDM_CUDA(h, cudaMemcpyAsync(d_bt, bt_h, (size_t)n_tb * n_tx * 8, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(d_br, br_h, (size_t)n_rb * n_w * 8, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(d_chan, chan, (size_t)r * L * 16, cudaMemcpyHostToDevice, d.stream));
    for (int b = 0; b < n_tb; ++b)
        build_tx_matrix<<<n_tx, 256, 0, d.stream>>>(d_T + (size_t)b * t_one, d_bt + (size_t)b * n_tx, N, sys->cp, n_tx);
    for (int a = 0; a < n_rb; ++a)
        build_rx_matrix<<<N, 256, 0, d.stream>>>(d_R + (size_t)a * r_one, d_br + (size_t)a * n_w, N, sys->tail_rx, sys->rm, sys->shift, n_rx, Kp);
    WOFDM_CUDA(h, cudaGetLastError());
    constexpr size_t smem = (size_t)(2 * BM * AS + 2 * BK * BS) * sizeof(double);
    WOFDM_CUDA(h, cudaFuncSetAttribute(gemm_power_f64<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const size_t mat = (size_t)2 * N * N;
    const dim3 g((n_var + 63) / 64, (n_var + 63) / 64);
    for (int v = 0; v < r; ++v) {
        // B_{b,ms} = H_ms(g_v) . Tx_mat(t_b) for every Tx basis window (channel v of d_chan: c0 = v)
        for (int b = 0; b < n_tb; ++b)
            build_b<false><<<dim3((N + 255) / 256, (Kp / 2 + BB - 1) / BB, Ms), 256, (size_t)(L + 2 * BB) * sizeof(double2), d.stream>>>(
                d_B + (size_t)b * Ms * Kp * N, d_T + (size_t)b * t_one, d_chan, L, N, n_tx, n_rx, n_rx, Kp, Ms, M, v, 1, k_isi);
        // X[a][b][ms] = Rbig(r_a) . B_{b,ms}: one stored contraction per Rx basis window over all Tx slices
        for (int a = 0; a < n_rb; ++a)
            gemm_power_f64<true><<<dim3(N / BN, 2 * N / BM, n_tb * Ms), 256, smem, d.stream>>>(
                d_R + (size_t)a * r_one, d_B, d_X + (size_t)a * n_tb * Ms * 2 * N * N, N, Kp, Ms, 0, 0, k_isi);
        WOFDM_CUDA(h, cudaGetLastError());
        h->launches += n_tb + n_rb + 1;
        if (H_out) {
            if (v == 0) gram_offdiag<false><<<n_var * (n_var + 1) / 2, 256, 0, d.stream>>>(d_X, d_H, n_var, N, n_tb);
            else gram_offdiag<true><<<n_var * (n_var + 1) / 2, 256, 0, d.stream>>>(d_X, d_H, n_var, N, n_tb);
        } else {
            // the parts, each one Gram product of the stored matrices (rows of pitch 2 mat: [slice 0 | ISI sum])
            zero_diag_kernel<<<n_var, 256, 0, d.stream>>>(d_X, n_var, N);
            for (int part = 0; part < 2; ++part) {
                double* const x = d_X + part * mat;
                double* const o = d_H + (size_t)part * n_var * n_var;
                if (v == 0) quad_eval_kernel<64, false><<<g, 256, 0, d.stream>>>(x, x, o, n_var, n_var, (int)mat, 0, 2 * mat, 2 * mat, 2.0);
                else quad_eval_kernel<64, true><<<g, 256, 0, d.stream>>>(x, x, o, n_var, n_var, (int)mat, 0, 2 * mat, 2 * mat, 2.0);
            }
            h->launches += 2;
        }
        WOFDM_CUDA(h, cudaGetLastError());
    }
    h->launches += n_tb + n_rb;
    if (H_out) {
        WOFDM_CUDA(h, cudaMemcpyAsync(H_out, d_H, (size_t)n_var * n_var * 8, cudaMemcpyDeviceToHost, d.stream));
    } else {
        WOFDM_CUDA(h, cudaMemcpyAsync(H_ici, d_H, (size_t)n_var * n_var * 8, cudaMemcpyDeviceToHost, d.stream));
        WOFDM_CUDA(h, cudaMemcpyAsync(H_isi, d_H + (size_t)n_var * n_var, (size_t)n_var * n_var * 8, cudaMemcpyDeviceToHost, d.stream));
    }
    WOFDM_CUDA(h, cudaEventRecord(h->hess_ev[1], d.stream));
    WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
    float ms = 0.f;
    h->hess_ms = cudaEventElapsedTime(&ms, h->hess_ev[0], h->hess_ev[1]) == cudaSuccess ? ms : -1.0;
    h->hess_passes = r;
    return WOFDM_OK;
}

// ---- the channel set as a few virtual channels --------------------------------------------------------------------------
// The Hessian is a Hermitian form in the taps: A0_u(h), AS_u(h) are linear in h, so H(h) = F(h h^H) with F linear, and
//     (1/C) sum_c H(h_c) = F(R) = sum_j H(g_j)   for R = (1/C) sum_c h_c h_c^H and ANY factor R = sum_j g_j g_j^H.
// C <= L: the channels themselves are that factor (weight 1/C on the result).  C > L: R (O(C L^2)) is factored by a
// pivoted Cholesky decomposition into r = rank(R) <= L columns g_j (weight 1): a set of 250 channels costs at most L passes.
// The decomposition stops when the largest remaining pivot (the variance left in the best unexplained tap) is at most
// kSetFactorTol times the largest diagonal entry of R, so the dropped remainder is a PSD matrix of trace at most
// L * kSetFactorTol * max_l R[l][l] -- below the fp64 rounding of the Gram sums for L <= 88.  Taps that are exact linear
// combinations of others (a rank-deficient set: repeated channels, a few propagation paths sinc-interpolated onto many
// taps) leave pivots at the rounding level and cost no pass.
constexpr double kSetFactorTol = 1e-14;

// chan: complex L x C column-major.  On return *virt points at r complex impulse responses of L taps (chan itself or fac)
// and *w is the weight of their summed Hessian.
static int channel_set_factor(wofdm_handle h, const double* chan, int L, int C, std::vector<double>& fac, const double** virt,
                              int* r, double* w) {
    for (size_t i = 0; i < (size_t)2 * L * C; ++i)
        if (!std::isfinite(chan[i])) return fail(h, WOFDM_EINVAL, "channel set: non-finite tap");
    if (C <= L) {
        *virt = chan; *r = C; *w = 1.0 / (double)C;
        return WOFDM_OK;
    }
    // R[i][j] = (1/C) sum_c h_c[i] conj(h_c[j]), row-major complex
    std::vector<double> R((size_t)2 * L * L, 0.0);
    for (int c = 0; c < C; ++c) {
        const double* hc = chan + (size_t)2 * L * c;
        for (int i = 0; i < L; ++i)
            for (int j = 0; j < L; ++j) {
                R[2 * ((size_t)i * L + j)] += hc[2 * i] * hc[2 * j] + hc[2 * i + 1] * hc[2 * j + 1];
                R[2 * ((size_t)i * L + j) + 1] += hc[2 * i + 1] * hc[2 * j] - hc[2 * i] * hc[2 * j + 1];
            }
    }
    for (double& x : R) x /= (double)C;
    // pivoted Cholesky: column k = (R[:, p] - sum_{j<k} g_j conj(g_j[p])) / sqrt(d_p), p the largest remaining diagonal
    std::vector<double> dg(L);
    std::vector<char> used(L, 0);
    double dmax = 0.0;
    for (int i = 0; i < L; ++i) { dg[i] = R[2 * ((size_t)i * L + i)]; dmax = std::max(dmax, dg[i]); }
    fac.assign((size_t)2 * L * L, 0.0);
    int k = 0;
    for (; k < L; ++k) {
        int p = -1;
        for (int i = 0; i < L; ++i)
            if (!used[i] && (p < 0 || dg[i] > dg[p])) p = i;
        if (!(dg[p] > kSetFactorTol * dmax)) break;
        const double s = std::sqrt(dg[p]);
        used[p] = 1;
        double* gk = fac.data() + (size_t)2 * L * k;
        for (int i = 0; i < L; ++i) {
            if (used[i]) continue;                          // pivots already taken (and p itself, set below)
            double re = R[2 * ((size_t)i * L + p)], im = R[2 * ((size_t)i * L + p) + 1];
            for (int j = 0; j < k; ++j) {                   // - g_j[i] conj(g_j[p])
                const double* gj = fac.data() + (size_t)2 * L * j;
                re -= gj[2 * i] * gj[2 * p] + gj[2 * i + 1] * gj[2 * p + 1];
                im -= gj[2 * i + 1] * gj[2 * p] - gj[2 * i] * gj[2 * p + 1];
            }
            gk[2 * i] = re / s; gk[2 * i + 1] = im / s;
            dg[i] -= gk[2 * i] * gk[2 * i] + gk[2 * i + 1] * gk[2 * i + 1];
        }
        gk[2 * p] = s;
    }
    *virt = fac.data(); *r = std::max(k, 1); *w = 1.0;         // (R = 0: one all-zero channel, H = 0)
    return WOFDM_OK;
}

// the reduced bases: columns of reduce_variable_tx / _rx (optimization_tools/utils.py:13-73) as full windows
static int reduced_bases(wofdm_handle h, const wofdm_sys_t* sys, std::vector<double>& bt, std::vector<double>& br) {
    const int n_tx = sys->N + sys->cp + sys->cs, n_w = sys->N + sys->tail_rx;
    const int n_tb = sys->tail_tx + 1, n_rb = sys->tail_rx / 2 + 1;
    bt.assign((size_t)n_tb * n_tx, 0.0);
    br.assign((size_t)n_rb * n_w, 0.0);
    std::vector<double> e(std::max(n_tb, n_rb));
    for (int b = 0; b < n_tb; ++b) {
        std::fill(e.begin(), e.end(), 0.0); e[b] = 1.0;
        int rc = wofdm_expand_window_tx(sys, e.data(), bt.data() + (size_t)b * n_tx);
        if (rc) return fail(h, rc, "expand_window_tx");
    }
    for (int a = 0; a < n_rb; ++a) {
        std::fill(e.begin(), e.end(), 0.0); e[a] = 1.0;
        int rc = wofdm_expand_window_rx(sys, e.data(), br.data() + (size_t)a * n_w);
        if (rc) return fail(h, rc, "expand_window_rx");
    }
    return WOFDM_OK;
}

// set = false: ONE impulse response (C = 1, no further checks); set = true: the mean over a set of C channels.
// H_out (the reduced-basis Hessian) or, with basis_tx / basis_rx given, the parts H_ici / H_isi.
static int window_hessian_run(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, int C, bool set,
                              const double* basis_tx, int n_tb, const double* basis_rx, int n_rb,
                              double* H_out, int* n_var_out, double* H_ici, double* H_isi) {
    if (!h) return WOFDM_EINVAL;
    int rc = validate_sys(h, sys, L);
    if (rc) return rc;
    const bool parts = H_out == nullptr;
    if (!parts && (!chan || !H_out)) return fail(h, WOFDM_EINVAL, "bad buffer");
    if (parts && (!chan || !basis_tx || !basis_rx || !H_ici || !H_isi || n_tb < 1 || n_rb < 1)) return fail(h, WOFDM_EINVAL, "bad buffer");
    if (set && C < 1) return fail(h, WOFDM_EINVAL, "channel set: C must be >= 1");
    if (sys->N % 64) return fail(h, WOFDM_EUNSUPPORTED, "interference path needs N to be a multiple of 64");
    if (parts && (size_t)2 * sys->N * sys->N % 16) return fail(h, WOFDM_EUNSUPPORTED, "N");
    std::vector<double> bt, br;
    if (!parts) {
        n_tb = sys->tail_tx + 1; n_rb = sys->tail_rx / 2 + 1;
        if (n_var_out) *n_var_out = n_tb * n_rb;
        rc = reduced_bases(h, sys, bt, br);
        if (rc) return rc;
        basis_tx = bt.data(); basis_rx = br.data();
    }
    const double* virt = chan;
    int r = 1;
    double w = 1.0;
    std::vector<double> fac;
    h->hess_factor_ms = 0.0;
    if (set) {
        const auto t0 = std::chrono::steady_clock::now();
        rc = channel_set_factor(h, chan, L, C, fac, &virt, &r, &w);
        if (rc) return rc;
        h->hess_factor_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    rc = window_hessian_core(h, sys, virt, L, r, basis_tx, n_tb, basis_rx, n_rb, H_out, H_ici, H_isi);
    if (rc || w == 1.0) return rc;
    const size_t nn = (size_t)n_tb * n_rb * n_tb * n_rb;
    for (double* H : {H_out, H_ici, H_isi})
        if (H)
            for (size_t i = 0; i < nn; ++i) H[i] *= w;
    return WOFDM_OK;
}

}  // namespace wofdm

using namespace wofdm;

extern "C" {

int wofdm_interf_power(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                       const double* chan, int L, int C, int mode, double* P) {
    return interf_run(h, sys, win_tx, win_rx, chan, L, C, mode, 0, P);
}

int wofdm_interf_power_scalar(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                              const double* chan, int L, int C, int mode, double* P) {
    return interf_run(h, sys, win_tx, win_rx, chan, L, C, mode, 1, P);
}

int wofdm_interf_last_timing(wofdm_handle h, double* total_ms, double* band_ms, double* gemm_ms, int* k_slice0, int* k_isi) {
    if (!h) return WOFDM_EINVAL;
    if (total_ms) *total_ms = h->interf_ms[0];
    if (band_ms) *band_ms = h->interf_ms[1];
    if (gemm_ms) *gemm_ms = h->interf_ms[2];
    if (k_slice0) *k_slice0 = (int)h->interf_kp;
    if (k_isi) *k_isi = (int)h->interf_k_isi;
    return WOFDM_OK;
}

int wofdm_window_hessian(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, double* H, int* n_var) {
    NvtxRange nvtx_("wofdm_window_hessian");
    return window_hessian_run(h, sys, chan, L, 1, false, nullptr, 0, nullptr, 0, H, n_var, nullptr, nullptr);
}

int wofdm_window_hessian_parts(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, const double* basis_tx, int n_tb,
                               const double* basis_rx, int n_rb, double* H_ici, double* H_isi) {
    NvtxRange nvtx_("wofdm_window_hessian_parts");
    return window_hessian_run(h, sys, chan, L, 1, false, basis_tx, n_tb, basis_rx, n_rb, nullptr, nullptr, H_ici, H_isi);
}

int wofdm_window_hessian_set(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, int C, double* H, int* n_var) {
    NvtxRange nvtx_("wofdm_window_hessian_set");
    return window_hessian_run(h, sys, chan, L, C, true, nullptr, 0, nullptr, 0, H, n_var, nullptr, nullptr);
}

int wofdm_window_hessian_parts_set(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, int C, const double* basis_tx,
                                   int n_tb, const double* basis_rx, int n_rb, double* H_ici, double* H_isi) {
    NvtxRange nvtx_("wofdm_window_hessian_parts_set");
    return window_hessian_run(h, sys, chan, L, C, true, basis_tx, n_tb, basis_rx, n_rb, nullptr, nullptr, H_ici, H_isi);
}

int wofdm_window_hessian_last_timing(wofdm_handle h, double* device_ms, double* factor_ms, int* passes) {
    if (!h) return WOFDM_EINVAL;
    if (device_ms) *device_ms = h->hess_ms;
    if (factor_ms) *factor_ms = h->hess_factor_ms;
    if (passes) *passes = h->hess_passes;
    return WOFDM_OK;
}

}  // extern "C"
