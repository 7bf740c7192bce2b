// interf_tf32.cu -- K2b', the interference contraction on 5th-generation tensor cores (tcgen05, kind::tf32)
// with a 3xTF32 split for fp32-grade accuracy (wofdm_interf_power mode 1).
//
//   [Re A; Im A] = Rbig . [Re B; Im B]       (interf.cu), one (channel, slice) = one 256-column block.
// Every fp64 operand x is split as x = hi + lo, hi = fp32(x) with the 13 low mantissa bits cleared (exactly a
// TF32 number), lo = fp32(x - hi) (the tensor core reads its top 19 bits); A.B ~ Ahi.Bhi + Ahi.Blo + Alo.Bhi,
// relative error ~2^-21 per product, accumulated in fp32 in tensor memory.
//
// A persistent CTA (192 threads, one per SM) works through 128 x 256 output tiles with TWO accumulators in TMEM (all
// 512 columns): the MMA issuer fills one while the four epilogue warps drain the other, so the tensor pipe does not
// idle through the epilogue, the TMEM allocation and the pipeline fill of every tile.  The hi/lo operands are
// stored in HBM PRE-TILED: every (row tile, K block of 32) is one contiguous block already in the canonical K-major
// no-swizzle UMMA layout (8-row x 16-byte core matrices; chunk c = (row/8)*64 + kchunk*8 + row%8 at byte 16*c), so a
// stage is filled by four cp.async.bulk copies (TMA engine, no tensor map) that complete on an mbarrier.
// Warp-specialised: one producer thread (bulk copies), one MMA thread (12 tcgen05.mma per K block = 4 K-steps x 3
// split terms, tcgen05.commit frees the stage), two stages.  Epilogue (four warps): tcgen05.ld the accumulator
// rows, mask the diagonal of slice 0, square, sum, one atomicAdd per row -- A itself is never written.
#include <algorithm>
#include "interf.h"

namespace wofdm {

namespace {

constexpr int TM = 128, TN = TF32_TN, KB = TF32_KB, NSTAGE = 2;
// Two CTAs that work on neighbouring row tiles of the same (channel, slice) form a thread-block cluster and share
// the B operand: each fetches one half of a B stage and MULTICASTS it into both shared memories.  Without it the
// persistent kernel pulls 96 KB per K block and SM out of L2 = 12.3 TB/s, which is the L2 limit, not the tensor pipe's.
constexpr int CLUSTER = 2;
constexpr int A_BYTES = TM * KB * 4, B_BYTES = TN * KB * 4;            // one hi (or lo) tile
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;                 // 96 KiB
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE: LBO = 128 B between the two 16-byte K chunks of one MMA, SBO = 1024 B between 8-row groups
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((128u >> 4) & 0x3fff) << 16;
    d |= (uint64_t)((1024u >> 4) & 0x3fff) << 32;
    d |= (uint64_t)1 << 46;                       // descriptor version of sm_100
    return d;
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
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
// the same copy delivered to the same offsets (data and mbarrier) of every CTA in `mask`
__device__ __forceinline__ void bulk_copy_multicast(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint16_t mask) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

}  // namespace

// Persistent: grid = CLUSTER * min(tile pairs, resident clusters) CTAs of 192 threads; cluster q takes the tile pairs
// q, q + clusters, ...; pair p = (slice p / (mtiles/2), row tiles 2*(p % (mtiles/2)) + rank).  Warps 0-3 = epilogue (TMEM lanes 32w..32w+31), warp 4 = producer, warp 5 = MMA issuer.
// Rt: [2N/TM][nk][hi|lo][TM*KB] tiles (tile_split_r below), Bt: [slices * N/TN][nk][hi|lo][TN*KB] tiles (build_b<true>, interf.cu)
constexpr int NTHREADS = 192;
__global__ void __launch_bounds__(NTHREADS, 1) gemm_power_tf32(const float* __restrict__ Rt, const float* __restrict__ Bt,
                                                              double* __restrict__ P, int N, int Kp, int Ms, int c0, int scalar,
                                                              int n_tiles, int nk_isi) {
    extern __shared__ __align__(1024) unsigned char sm[];
    __shared__ __align__(8) unsigned long long full_bar[NSTAGE], empty_bar[NSTAGE], acc_full[2], acc_empty[2];
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr uint16_t CL_MASK = (1u << CLUSTER) - 1u;
    const int nk = Kp / KB, mtiles = 2 * N / TM;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int q0 = blockIdx.x / CLUSTER, nq = gridDim.x / CLUSTER, n_pairs = n_tiles / CLUSTER, ppairs = mtiles / CLUSTER;
    const int ntile = N / TN;                                  // column tiles per slice: B tile sv = s * ntile + nt

    if (warp == 4) {   // both accumulators: all 512 columns (one CTA per SM: the stages take 192 KB of shared memory)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tmem_base_s)), "r"(2 * TN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < NSTAGE; ++i) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&full_bar[i])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(&empty_bar[i])), "r"(CLUSTER) : "memory");   // released by every CTA's MMAs
        }
        for (int i = 0; i < 2; ++i) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(&acc_full[i])) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" :: "r"(smem_u32(&acc_empty[i])) : "memory");   // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();                           // the peer's barriers exist before anything is multicast onto them
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base_s;

    if (warp == 4) {
        if (lane == 0) {
            // ===== producer: two bulk copies per stage, K blocks numbered through all of this CTA's tiles =====
            int it = 0;
            for (int p = q0; p < n_pairs; p += nq) {
                const float* ra = Rt + (size_t)((p % ppairs) * CLUSTER + rank) * nk * (2 * TM * KB);
                const float* rb = Bt + (size_t)(p / ppairs) * nk * (2 * TN * KB);
                const int nk_t = ((p / ppairs / ntile) % Ms) == 0 ? nk : nk_isi; // ISI slices: non-zero K prefix only
                for (int kb = 0; kb < nk_t; ++kb, ++it) {
                    const int st = it % NSTAGE;
                    if (it >= NSTAGE) mbar_wait(smem_u32(&empty_bar[st]), (uint32_t)(((it / NSTAGE) - 1) & 1));
                    const uint32_t bar = smem_u32(&full_bar[st]), dst = smem_u32(sm + (size_t)st * STAGE_BYTES);
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"((uint32_t)STAGE_BYTES) : "memory");
                    bulk_copy(dst, ra + (size_t)kb * (2 * TM * KB), 2 * A_BYTES, bar);                 // A hi | lo
                    // B hi | lo: this CTA's share, delivered to every CTA of the cluster (each receives all of it)
                    constexpr uint32_t QB = 2 * B_BYTES / CLUSTER;
                    bulk_copy_multicast(dst + 2 * A_BYTES + rank * QB,
                                        reinterpret_cast<const unsigned char*>(rb + (size_t)kb * (2 * TN * KB)) + (size_t)rank * QB, QB, bar, CL_MASK);
                }
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {
            // ===== MMA issuer: tile tl accumulates into TMEM columns [(tl & 1) * TN, +TN) while the epilogue drains the other half =====
            int it = 0, tl = 0;
            for (int p = q0; p < n_pairs; p += nq, ++tl) {
                const int buf = tl & 1;
                if (tl >= 2) {
                    mbar_wait(smem_u32(&acc_empty[buf]), (uint32_t)(((tl >> 1) - 1) & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                const uint32_t tacc = tmem + (uint32_t)(buf * TN);
                const int nk_t = ((p / ppairs / ntile) % Ms) == 0 ? nk : nk_isi;
                for (int kb = 0; kb < nk_t; ++kb, ++it) {
                    const int st = it % NSTAGE;
                    mbar_wait(smem_u32(&full_bar[st]), (uint32_t)((it / NSTAGE) & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_hi = smem_u32(sm + (size_t)st * STAGE_BYTES), a_lo = a_hi + A_BYTES, b_hi = a_hi + 2 * A_BYTES, b_lo = b_hi + B_BYTES;
#pragma unroll
                    for (int j = 0; j < KB / 8; ++j) {                             // one MMA consumes 8 TF32 = two 16-byte chunks
                        const uint32_t off = (uint32_t)j * 256u;
                        mma_tf32(tacc, umma_desc(a_hi + off), umma_desc(b_hi + off), (kb | j) != 0);
                        mma_tf32(tacc, umma_desc(a_hi + off), umma_desc(b_lo + off), 1u);
                        mma_tf32(tacc, umma_desc(a_lo + off), umma_desc(b_hi + off), 1u);
                    }
                    // frees stage st in every CTA of the cluster (each of them multicasts into it)
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                                 :: "r"(smem_u32(&empty_bar[st])), "h"(CL_MASK) : "memory");
                }
                // completes once per tile, after every MMA of the tile
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(&acc_full[buf])) : "memory");
            }
        }
    } else {
        // ===== epilogue warps: thread = one row of the tile (TMEM lane 32*warp + lane) =====
        int tl = 0;
        for (int p = q0; p < n_pairs; p += nq, ++tl) {
            const int buf = tl & 1;
            const int m0 = ((p % ppairs) * CLUSTER + (int)rank) * TM, sv = p / ppairs, s = sv / ntile, j0 = (sv % ntile) * TN;
            mbar_wait(smem_u32(&acc_full[buf]), (uint32_t)((tl >> 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int r = m0 + warp * 32 + lane, k = r % N;
            const int c = c0 + s / Ms, ms = s % Ms;
            float pw = 0.f;
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
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float x = __uint_as_float(v[i]);
                    if (!(ms == 0 && j0 + cc * 32 + i == k)) pw = fmaf(x, x, pw);
                }
            }
            // this warp's quarter of the accumulator has been read: hand the buffer back to the MMA issuer
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(&acc_empty[buf])) : "memory");
            atomicAdd(scalar ? &P[c] : &P[(size_t)c * N + k], (double)pw);
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();                           // nobody leaves while the peer's releases can still land on its barriers
    if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(2 * TN) : "memory");
}

__device__ __forceinline__ void split_hi_lo(double x, float& hi, float& lo) {
    hi = __uint_as_float(__float_as_uint((float)x) & 0xffffe000u);
    lo = (float)(x - (double)hi);
}
// offset (in floats) of element (row, kk) inside its [hi|lo] tile pair: tile = (row/rows_per_tile, kk/KB)
__device__ __forceinline__ size_t tiled_off(int row, int kk, int rows_per_tile, int nk) {
    const int rt = row / rows_per_tile, r = row % rows_per_tile, kb = kk / KB, k = kk % KB;
    const int c = (r >> 3) * 64 + (k >> 2) * 8 + (r & 7);
    return ((size_t)rt * nk + kb) * (2 * (size_t)rows_per_tile * KB) + (size_t)c * 4 + (k & 3);
}

// Rbig [2N][Kp] fp64 -> Rt tiles (tiny: 2N x Kp elements)
__global__ void tile_split_r(const double* __restrict__ Rbig, float* __restrict__ Rt, int rows, int Kp) {
    const int nk = Kp / KB;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)rows * Kp; i += (size_t)gridDim.x * blockDim.x) {
        const int row = (int)(i / Kp), kk = (int)(i % Kp);
        float hi, lo;
        split_hi_lo(Rbig[i], hi, lo);
        const size_t o = tiled_off(row, kk, TM, nk);
        Rt[o] = hi;
        Rt[o + (size_t)TM * KB] = lo;
    }
}

float* interf_tf32_b_tiles(const InterfDev& v, int N) { return v.tf32_work + (size_t)2 * 2 * N * v.Kp; }

int interf_gemm_tf32(wofdm_ctx* h, const wofdm_sys_t* sys, const InterfDev& v, int Ms, int c0, int slices, int scalar,
                     int k_isi) {
    DeviceCtx& d = h->devs[0];
    const int N = sys->N;
    if (N % TN) return fail(h, WOFDM_EUNSUPPORTED, "TF32-split interference path needs N to be a multiple of 256");
    if (v.Kp % KB) return fail(h, WOFDM_EINVAL, "Kp must be a multiple of 32");
    const size_t nr = (size_t)2 * 2 * N * v.Kp;                      // Rt: hi + lo
    // fp32 work buffers live behind the fp64 B matrix of this batch (interf_upload reserved room for them)
    float* Rt = v.tf32_work;
    float* Bt = Rt + nr;
    tile_split_r<<<128, 256, 0, d.stream>>>(v.Rbig, Rt, 2 * N, v.Kp);
    const int nk_isi = k_isi / KB;

    WOFDM_CUDA(h, cudaGetLastError());
    const size_t smem = (size_t)NSTAGE * STAGE_BYTES;
    const int n_tiles = (2 * N / TM) * slices * (N / TN);
    WOFDM_CUDA(h, cudaFuncSetAttribute(gemm_power_tf32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(CLUSTER * d.sm_count); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = d.stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int ncl = 0;
    WOFDM_CUDA(h, cudaOccupancyMaxActiveClusters(&ncl, gemm_power_tf32, &cfg));
    if (ncl < 1) return fail(h, WOFDM_EUNSUPPORTED, "no cluster of the TF32 contraction kernel fits the device");
    static_assert((2 * TN / TM) % CLUSTER == 0, "row tiles pair up inside a cluster");
    cfg.gridDim = dim3(CLUSTER * std::min(n_tiles / CLUSTER, ncl));
    WOFDM_CUDA(h, cudaLaunchKernelEx(&cfg, gemm_power_tf32, (const float*)Rt, (const float*)Bt, v.P, N, v.Kp, Ms, c0, scalar, n_tiles, nk_isi));
    WOFDM_CUDA(h, cudaGetLastError());
    h->launches += 2;
    return WOFDM_OK;
}

}  // namespace wofdm
