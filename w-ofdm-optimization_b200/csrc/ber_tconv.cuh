// ber_tconv.cuh -- the pieces of K1's channel convolution on the 5th-generation tensor cores (tcgen05, sm_100a) that the
// frame kernel of ber_tconv2.cuh builds on: the Hankel operand, its fp16 split, its scales, and the tcgen05 wrappers.
//
// The L-tap tapped-delay-line convolution r = conv(h, u) (wofdm_simulation.py:206, main_BER_calculation.m:260) is a
// tensor-core product whose A operand is the frame stream itself:
//
//   * every stream sample is split in two fp16 pairs, u = hi + lo (|u - hi - lo| <= 2^-22 |u|), stored as half2 words
//     (re, im) in two arrays ahi[], alo[];
//   * row r of the operand is the 24 samples 4r-20 .. 4r+3 (K = 48 halves).  Rows are 16 bytes apart -- exactly the
//     pitch of the rows inside an 8 x 16-byte core matrix of the K-major, no-swizzle UMMA layout -- so the raw array IS
//     a canonical operand of the (overlapping) Hankel matrix: LBO = 16 B (next K chunk = next 4 samples), SBO = 128 B
//     (next 8 rows).  Nothing is gathered or copied;
//   * B (16 x 48, K-major) holds the taps, rebuilt per frame: output column 2o / 2o+1 = Re / Im of r[4 row + o], o < 4, from
//     T_hi; columns 8 + (2o, 2o+1) the same from T_lo.  r = hi.[T_hi | T_lo] + lo.[T_hi | 0]: two 128 x 16 x 16 MMAs per
//     (tile of 512 samples, K step of 8 samples), fp32 accumulation in tensor memory (16 columns per tile).
#pragma once
#include <cuda_fp16.h>
#include "ber_kernel.cuh"

namespace wofdm {

constexpr int TCV_LB = 21;            // taps of the Hankel operand (row r = samples 4r - (LB-1) .. 4r + 3)
constexpr float TCV_XSCALE = 64.0f;   // stream and taps are scaled by powers of two into the comfortable fp16 range;
constexpr float TCV_HSCALE = 16.0f;   // everything behind the channel is scale-invariant (measured powers, pilot equaliser)
// tensor-memory columns a CTA allocates: 16 per tile, a power of two (two CTAs per SM when 256 are enough)
__host__ __device__ constexpr uint32_t tconv_tmem_cols(int ntile) { return 16 * ntile <= 256 ? 256u : 512u; }

__device__ __forceinline__ uint32_t tcv_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t tcv_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((lbo >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;                       // descriptor version of sm_100
    return d;
}
__device__ __forceinline__ void tcv_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    constexpr uint32_t idesc = (1u << 4) | ((16u >> 3) << 17) | ((128u >> 4) << 24);   // D f32, A = B = f16, K-major, N 16, M 128
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tcv_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (int it = 0; it < (1 << 22) && !done; ++it)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (!done) __trap();                          // never spin forever on a GPU we share
}
// four accumulator columns of this thread's row (TMEM lane) as two complex numbers
__device__ __forceinline__ void tcv_ld4(uint32_t taddr, float2& a, float2& b) {
    uint32_t v0, v1, v2, v3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3) : "r"(taddr) : "memory");
    a = make_float2(__uint_as_float(v0), __uint_as_float(v1));
    b = make_float2(__uint_as_float(v2), __uint_as_float(v3));
}
// eight / sixteen accumulator columns of this thread's row
__device__ __forceinline__ void tcv_ld8(uint32_t taddr, float2& a, float2& b, float2& c, float2& d) {
    uint32_t v[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr) : "memory");
    a = make_float2(__uint_as_float(v[0]), __uint_as_float(v[1]));
    b = make_float2(__uint_as_float(v[2]), __uint_as_float(v[3]));
    c = make_float2(__uint_as_float(v[4]), __uint_as_float(v[5]));
    d = make_float2(__uint_as_float(v[6]), __uint_as_float(v[7]));
}
__device__ __forceinline__ void tcv_ld16(uint32_t taddr, float2 (&c)[8]) {
    uint32_t v[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = make_float2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
}
__device__ __forceinline__ bool tcv_elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t h2_bits(__half2 h) { return *reinterpret_cast<const uint32_t*>(&h); }
__device__ __forceinline__ __half2 bits_h2(uint32_t w) { return *reinterpret_cast<const __half2*>(&w); }
// u = hi + lo.  The residual v - hi comes from the mixed-precision FMA (fp16 x fp16 + fp32, SASS FHFMA): hi * (-1) + v with
// one rounding = the fp32 difference, one instruction per component instead of unpack + subtract.
__device__ __forceinline__ void split_h2(float2 v, uint32_t& hi, uint32_t& lo) {
    const __half2 a = __floats2half2_rn(v.x, v.y);
    hi = h2_bits(a);
    const unsigned short al = (unsigned short)(hi & 0xffffu), ah = (unsigned short)(hi >> 16), mone = 0xbc00u;   // -1.0
    float dx, dy;
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(dx) : "h"(al), "h"(mone), "f"(v.x));
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(dy) : "h"(ah), "h"(mone), "f"(v.y));
    lo = h2_bits(__floats2half2_rn(dx, dy));
}
__device__ __forceinline__ float2 join_h2(uint32_t hi, uint32_t lo) { return add2(__half22float2(bits_h2(hi)), __half22float2(bits_h2(lo))); }

}  // namespace wofdm
