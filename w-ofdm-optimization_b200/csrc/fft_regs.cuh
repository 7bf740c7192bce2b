// fft_regs.cuh -- register-resident Stockham FFT, 16 points per thread, N/16 threads per transform.
//
// N = 16^a * r (r in {1,2,4,8}): `a` radix-16 passes (each a 4x4 DFT in registers) and, if r > 1,
// one final radix-r pass on the same 16 registers.  Between passes the N points are transposed
// through a padded shared-memory buffer (index i -> i + i/16, conflict-free for 8- and 16-byte
// elements).  Thread t of a transform holds points t + q*(N/16), q = 0..15, on entry AND on exit
// (natural order), which is the layout symbol generation, CP/CS insertion and the equaliser use.
//
// Twiddles come from a table built on the host in double precision (see fft_twiddle_count):
//   section P_1 (a >= 2),     entry [k*TW1_PITCH + m] = exp(-2*pi*i * k*m / 256),  k < 16, m < 16 (a thread's 15 factors are one row)
//   section P_2 (a >= 3),     entry [m*256 + k] = exp(-2*pi*i * k*m / 4096),       m < 16, k < 256
//   section F   (if r > 1),   entry [m*(N/r) + j] = exp(-2*pi*i * j*m / N),       m < r,  j < N/r
// DIR = -1 forward (unscaled), DIR = +1 inverse (unscaled; the caller folds 1/N into the Tx window).
// Replaces the dense IDFT/DFT products of the reference (python/ofdm_utils/transmitter.py:38-58,
// receiver.py:113-133; matlab dftmtx at main_BER_calculation.m:306,370).
#pragma once
#include "common.cuh"

namespace wofdm {

constexpr int TW1_PITCH = 18;     // row pitch of the first twiddle section (16 entries + 2: rows 144 B apart, 128-bit loads without bank conflicts)
template <int N> struct FftPlan {
    static constexpr int a = (N % 4096 == 0) ? 3 : (N % 256 == 0) ? 2 : (N % 16 == 0) ? 1 : 0;
    static constexpr int p16 = (a == 3) ? 4096 : (a == 2) ? 256 : (a == 1) ? 16 : 1;
    static constexpr int r = N / p16;
    static constexpr int TPF = N / 16;                 // threads per transform
    static constexpr int XLEN = N + N / 8;             // padded exchange buffer (elements)
    static constexpr int NTW = ((a >= 2) ? 16 * TW1_PITCH : 0) + ((a >= 3) ? 4096 : 0) + ((r > 1) ? N : 0);
    static_assert(N >= 16 && (N & (N - 1)) == 0 && N <= 4096, "N must be a power of two in [16, 4096]");
    static_assert(r == 1 || r == 2 || r == 4 || r == 8, "unsupported factorisation");
};

// two pad elements per 16: a thread's 16 consecutive points of the first exchange start 16-byte aligned (vector stores),
// and both the stores (lane stride 18) and the transposed loads (lane stride 1) stay free of bank conflicts
__host__ __device__ constexpr int fft_pad(int i) { return i + 2 * (i >> 4); }

// multiply by exp(DIR * 2*pi*i * E / 16), E compile time
template <typename T, int DIR, int E> __device__ __forceinline__ V2<T> mul_w16(V2<T> a) {
    constexpr int e = ((E % 16) + 16) % 16;
    constexpr T C1 = (T)0.92387953251128673848, S1 = (T)0.38268343236508978178, R2 = (T)0.70710678118654752440;
    if constexpr (e == 0) return a;
    else if constexpr (e == 8) return mk2<T>(-a.x, -a.y);
    else if constexpr (e == 4) return DIR > 0 ? rotj(a) : rotmj(a);
    else if constexpr (e == 12) return DIR > 0 ? rotmj(a) : rotj(a);
    else if constexpr (e == 2 || e == 6 || e == 10 || e == 14) {
        // R2 * (sc + i ss) * a = R2 * (sc*a + ss*(i a)), sc, ss = +-1
        constexpr bool sc_pos = (e == 2 || e == 14);
        constexpr bool ss_pos0 = (e == 2 || e == 6);
        constexpr bool ss_pos = DIR > 0 ? ss_pos0 : !ss_pos0;
        const V2<T> u = sc_pos ? a : mk2<T>(-a.x, -a.y);
        const V2<T> w = ss_pos ? rotj(a) : rotmj(a);
        return cscale(R2, cadd(u, w));
    } else {
        constexpr T ctab[16] = {1, C1, R2, S1, 0, -S1, -R2, -C1, -1, -C1, -R2, -S1, 0, S1, R2, C1};
        constexpr T stab[16] = {0, S1, R2, C1, 1, C1, R2, S1, 0, -S1, -R2, -C1, -1, -C1, -R2, -S1};
        constexpr T c = ctab[e];
        constexpr T s = DIR > 0 ? stab[e] : -stab[e];
        return cmul(a, mk2<T>(c, s));
    }
}

template <typename T, int DIR> __device__ __forceinline__ void bfly2(V2<T>& a0, V2<T>& a1) {
    const V2<T> s = cadd(a0, a1), d = csub(a0, a1);
    a0 = s; a1 = d;
}

template <typename T, int DIR> __device__ __forceinline__ void bfly4(V2<T>& a0, V2<T>& a1, V2<T>& a2, V2<T>& a3) {
    const V2<T> s02 = cadd(a0, a2), d02 = csub(a0, a2), s13 = cadd(a1, a3), d13 = csub(a1, a3);
    a0 = cadd(s02, s13);
    a2 = csub(s02, s13);
    if constexpr (DIR < 0) {  // X1 = d02 - i d13, X3 = d02 + i d13
        a1 = cadd(d02, rotmj(d13));
        a3 = cadd(d02, rotj(d13));
    } else {
        a1 = cadd(d02, rotj(d13));
        a3 = cadd(d02, rotmj(d13));
    }
}

// 8-point DFT on x[0..7] (natural order in and out)
template <typename T, int DIR> __device__ __forceinline__ void dft8(V2<T> (&x)[8]) {
    bfly4<T, DIR>(x[0], x[2], x[4], x[6]);   // E[k] in x[0],x[2],x[4],x[6]
    bfly4<T, DIR>(x[1], x[3], x[5], x[7]);   // O[k] in x[1],x[3],x[5],x[7]
    const V2<T> o0 = x[1], o1 = mul_w16<T, DIR, 2>(x[3]), o2 = mul_w16<T, DIR, 4>(x[5]), o3 = mul_w16<T, DIR, 6>(x[7]);
    const V2<T> e0 = x[0], e1 = x[2], e2 = x[4], e3 = x[6];
    x[0] = cadd(e0, o0); x[4] = csub(e0, o0);
    x[1] = cadd(e1, o1); x[5] = csub(e1, o1);
    x[2] = cadd(e2, o2); x[6] = csub(e2, o2);
    x[3] = cadd(e3, o3); x[7] = csub(e3, o3);
}

// 16-point DFT, natural order in and out: n = 4*n1 + n2, k = k1 + 4*k2
template <typename T, int DIR> __device__ __forceinline__ void dft16(V2<T> (&v)[16]) {
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) bfly4<T, DIR>(v[n2], v[n2 + 4], v[n2 + 8], v[n2 + 12]);
    // v[n2 + 4*k1] *= W16^(k1*n2)
    v[5] = mul_w16<T, DIR, 1>(v[5]);   v[6] = mul_w16<T, DIR, 2>(v[6]);   v[7] = mul_w16<T, DIR, 3>(v[7]);
    v[9] = mul_w16<T, DIR, 2>(v[9]);   v[10] = mul_w16<T, DIR, 4>(v[10]); v[11] = mul_w16<T, DIR, 6>(v[11]);
    v[13] = mul_w16<T, DIR, 3>(v[13]); v[14] = mul_w16<T, DIR, 6>(v[14]); v[15] = mul_w16<T, DIR, 9>(v[15]);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) bfly4<T, DIR>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
    // v[4*k1 + k2] holds X[k1 + 4*k2]: transpose the 4x4 register tile
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i + 1; j < 4; ++j) { const V2<T> tmp = v[4 * i + j]; v[4 * i + j] = v[4 * j + i]; v[4 * j + i] = tmp; }
}

template <typename T, int DIR> __device__ __forceinline__ V2<T> tw_apply(V2<T> a, V2<T> w) {
    if constexpr (DIR < 0) return cmul(a, w);
    else return cmulc(a, w);
}

// Barrier between the threads of one transform: the N/16 threads of a group sit in one warp when
// N <= 512 (groups are aligned to their size), so a warp barrier is enough and the CTA's other
// warps run on; larger transforms span warps and use the CTA barrier.
// N = 1024: a transform spans two warps; with at most 15 transforms per CTA (NB) each group gets its own
// named barrier (ids 1..NB, TPF threads) instead of stalling the whole CTA.
template <int TPF, int NB> __device__ __forceinline__ void fft_group_sync(int group) {
    if constexpr (TPF <= 32) __syncwarp();
    else if constexpr (NB >= 1 && NB <= 15) asm volatile("bar.sync %0, %1;" :: "r"(group + 1), "n"(TPF) : "memory");
    else __syncthreads();
}

// 16 consecutive complex values, 16-byte aligned: 128-bit accesses (eight for float2, one per element for double2)
__device__ __forceinline__ void store16(float2* dst, const float2 (&v)[16]) {
    float4* d = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = make_float4(v[2 * i].x, v[2 * i].y, v[2 * i + 1].x, v[2 * i + 1].y);
}
__device__ __forceinline__ void store16(double2* dst, const double2 (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) dst[i] = v[i];
}
__device__ __forceinline__ void load16(float2 (&w)[16], const float2* src) {
    const float4* s = reinterpret_cast<const float4*>(src);
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float4 q = s[i]; w[2 * i] = make_float2(q.x, q.y); w[2 * i + 1] = make_float2(q.z, q.w); }
}
__device__ __forceinline__ void load16(double2 (&w)[16], const double2* src) {
#pragma unroll
    for (int i = 0; i < 16; ++i) w[i] = src[i];
}

// One transform per group of N/16 threads; EVERY thread of the CTA must call this (it contains
// barriers).  xb: this group's exchange buffer (FftPlan<N>::XLEN elements, shared memory), private
// to the group; tw: twiddle table (FftPlan<N>::NTW elements).  Memory that aliases xb and is
// touched by OTHER groups needs a __syncthreads() of the caller on both sides of this call.
// NB / group: number of transforms the CTA runs side by side and this thread's transform (for the named barriers).
template <typename T, int N, int DIR, int NB = 0>
__device__ __forceinline__ void fft_regs(V2<T> (&v)[16], const int t, V2<T>* __restrict__ xb,
                                         const V2<T>* __restrict__ tw, const int group = 0) {
    using P = FftPlan<N>;
    constexpr int TPF = P::TPF;
    int tw_off = 0;
#pragma unroll
    for (int p = 0; p < P::a; ++p) {
        const int Ns = (p == 0) ? 1 : (p == 1) ? 16 : 256;
        const int k = t & (Ns - 1);
        if (p > 0) {
            fft_group_sync<TPF, NB>(group);
            {   // fft_pad(t + m TPF) = fft_pad(t) + m (TPF + TPF/8): one address, immediate offsets
                const V2<T>* const xr = xb + fft_pad(t);
#pragma unroll
                for (int m = 0; m < 16; ++m) v[m] = xr[m * (TPF + TPF / 8)];
            }
            V2<T> w[16];
            if (p == 1) {                 // (not held across the exchange: the kernels around this are register bound)
                load16(w, tw + tw_off + k * TW1_PITCH);
            } else {
#pragma unroll
                for (int m = 1; m < 16; ++m) w[m] = tw[tw_off + m * Ns + k];
            }
#pragma unroll
            for (int m = 1; m < 16; ++m) v[m] = tw_apply<T, DIR>(v[m], w[m]);
            tw_off += p == 1 ? 16 * TW1_PITCH : 16 * Ns;
        }
        dft16<T, DIR>(v);
        const bool last = (p == P::a - 1);
        if (!(last && P::r == 1)) {
            fft_group_sync<TPF, NB>(group);        // the group has finished reading the previous layout (also of an earlier call)
            const int base = (t - k) * 16 + k;
            {   // base = 16 Ns j + k, k < Ns: fft_pad(base + m Ns) = fft_pad(base) + m (Ns = 1) or + m (Ns + Ns/8)
                V2<T>* const xw = xb + fft_pad(base);
                if (Ns == 1) {
                    store16(xw, v);           // 16 consecutive points, 16-byte aligned: vector stores
                } else {
                    const int step = Ns + Ns / 8;
#pragma unroll
                    for (int m = 0; m < 16; ++m) xw[m * step] = v[m];
                }
            }
        }
    }
    if constexpr (P::r > 1) {
        constexpr int r = P::r, G = 16 / r;   // G butterflies of radix r per thread
        fft_group_sync<TPF, NB>(group);
        if constexpr (TPF % 16 == 0) {
            const V2<T>* const xr = xb + fft_pad(t);
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = xr[q * (TPF + TPF / 8)];
        } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = xb[fft_pad(t + q * TPF)];
        }
#pragma unroll
        for (int b = 0; b < G; ++b) {
            const int jb = t + b * TPF;
#pragma unroll
            for (int m = 1; m < r; ++m) v[b + m * G] = tw_apply<T, DIR>(v[b + m * G], tw[tw_off + m * (N / r) + jb]);
            if constexpr (r == 2) {
                bfly2<T, DIR>(v[b], v[b + G]);
            } else if constexpr (r == 4) {
                bfly4<T, DIR>(v[b], v[b + G], v[b + 2 * G], v[b + 3 * G]);
            } else {
                V2<T> x[8];
#pragma unroll
                for (int m = 0; m < 8; ++m) x[m] = v[b + m * G];
                dft8<T, DIR>(x);
#pragma unroll
                for (int m = 0; m < 8; ++m) v[b + m * G] = x[m];
            }
        }
    }
}

}  // namespace wofdm
