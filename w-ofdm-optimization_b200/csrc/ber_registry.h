// ber_registry.h -- host-side table of the compiled K1 variants.
#pragma once
#include <cuda_runtime.h>
#include <tuple>
#include <vector>
#include "ber_kernel.cuh"

namespace wofdm {

struct BerVariant {
    const char* name;
    int N, NT, TC, LB, MINB;
    int CL;                    // CTAs per frame (thread-block cluster size)
    bool circ;                 // interior of the channel output as a circular convolution (needs a flat Tx window)
    bool txs = false;          // ber_kernel.cuh TXS: reads BerParams::tx_stream (channel-mask variant); the staged kernels always do
    bool full;                 // every register of every thread is a live stream sample (NT*TC == S*stride)
    int ntile;                 // > 0: channel convolution on the tensor cores (ber_tconv2.cuh), frames of up to 512*ntile samples
    int launch_threads;        // threads per CTA at launch (NT, plus the MMA warp of ber_tconv2.cuh)
    bool txy = false;          // ber_tconv2.cuh: takes the Tx stream from the mask product's output (BerParams::tx_y) and nothing else
    bool res = false;          // counters resolved by sub-carrier / channel (BerParams::res_bins / res_chan) and nothing else
    bool fixed_shape = false;  // ber_tconv2.cuh HS: the switches of one shape class as constants (ber_host.cu: tconv2_fixed_shape)
    int geom = 0;              // > 0: ... and the geometry tconv2_geom(geom) as constants (ber_host.cu: tconv2_fixed_geometry)
    bool fp64, verify;
    BerSmem (*layout)(int S, int stride, int tail_tx, int tail_rx, int L, int chunk, int use_global);
    const void* fn;
    cudaError_t (*launch)(const BerParams& prm, int grid, size_t smem, cudaStream_t st);
    // the template arguments that fix the arithmetic and the noise blocks: a kernel and its resolved-counter twin (res) have
    // the same key
    auto key() const { return std::tie(fp64, N, NT, TC, LB, MINB, CL, circ, full, txs, txy); }
};

// grid = CTAs of THREADS threads (a multiple of CL); CL > 1 launches thread-block clusters of CL CTAs
template <auto KERNEL, int THREADS, int CL>
cudaError_t launch_frames(const BerParams& prm, int grid, size_t smem, cudaStream_t st) {
    if constexpr (CL == 1) {
        KERNEL<<<grid, THREADS, smem, st>>>(prm);
        return cudaGetLastError();
    } else {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, KERNEL, prm);
    }
}

template <typename T, int N, int NT, int TC, int LB, int MINB, bool FULL, bool V, int CL = 1, bool CIRC = false, bool TXS = false,
          bool RES = false>
struct BerVariantImpl {
    static BerVariant make(const char* name) {
        constexpr auto kernel = &ber_frame_kernel<T, N, NT, TC, LB, MINB, FULL, V, CL, CIRC, TXS, RES>;
        BerVariant v;
        v.name = name; v.N = N; v.NT = NT; v.TC = TC; v.LB = LB; v.MINB = MINB; v.CL = CL; v.circ = CIRC; v.txs = TXS || TC == 0; v.full = FULL; v.ntile = 0; v.launch_threads = NT;
        v.fp64 = sizeof(T) == 8; v.verify = V; v.res = RES;
        v.layout = &ber_smem_layout<T, N, NT, TC, LB, RES>;
        v.fn = reinterpret_cast<const void*>(kernel);
        v.launch = &launch_frames<kernel, NT, CL>;
        return v;
    }
};

// ber_frame_kernel<T, N, NT, TC, LB, MINB, FULL, ...> registered as "ber_<tag>_n<N>_t<NT>_c<TC>_l<LB>_b<MINB>_f<FULL><sfx>";
// "..." are the template arguments from V on (V = verify instance, CL, CIRC, TXS, RES)
#define WOFDM_VARIANT(tag, sfx, T, N, NT, TC, LB, MINB, FULL, ...)                                    \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, __VA_ARGS__>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL sfx));

void register_ber_f32_staged(std::vector<BerVariant>& out);
void register_ber_f32_tconv2(std::vector<BerVariant>& out);
void register_ber_f32_tconv2_hs(std::vector<BerVariant>& out);       // ... its fixed-shape instances
void register_ber_f64_staged(std::vector<BerVariant>& out);
void register_ber_f32_regs(std::vector<BerVariant>& out);
void register_ber_f32_regs_big(std::vector<BerVariant>& out);
void register_ber_f32_tconv2_res(std::vector<BerVariant>& out);      // resolved counters (RES): tensor-core ...
void register_ber_f32_tconv2_res_big(std::vector<BerVariant>& out);
void register_ber_staged_res(std::vector<BerVariant>& out);          // ... staged ...
void register_ber_f32_regs_res(std::vector<BerVariant>& out);        // ... and register policies
void register_ber_f32_tconv2_txy_res(std::vector<BerVariant>& out); // the channel-mask chain's twins: tensor-core gather ...
void register_ber_f32_regs_txs_res(std::vector<BerVariant>& out);    // ... and register kernels on the assembled stream

}  // namespace wofdm
