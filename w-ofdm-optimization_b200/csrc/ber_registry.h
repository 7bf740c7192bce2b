// ber_registry.h -- host-side table of the compiled K1 variants.
#pragma once
#include <cuda_runtime.h>
#include <vector>
#include "ber_kernel.cuh"

namespace wofdm {

struct BerVariant {
    const char* name;
    int N, NT, TC, LB, MINB;
    int CL;                    // CTAs per frame (thread-block cluster size)
    bool circ;                 // interior of the channel output as a circular convolution (needs a flat Tx window)
    bool txs;                  // accepts BerParams::tx_stream (channel-mask variant); the staged kernels always do
    bool full;                 // every register of every thread is a live stream sample (NT*TC == S*stride)
    int ntile;                 // > 0: channel convolution on the tensor cores (ber_tconv*.cuh), frames of up to 512*ntile samples
    int launch_threads;        // threads per CTA at launch (NT, plus the MMA warp of ber_tconv2.cuh)
    int gen;                   // tensor-core kernels: 1 = ber_tconv.cuh (64-bit noise draws by position), 2 = ber_tconv2.cuh (48-bit draws)
    bool txy = false;          // ber_tconv2.cuh: takes the Tx stream from the mask product's output (BerParams::tx_y) and nothing else
    bool res = false;          // counters resolved by sub-carrier / channel (BerParams::res_bins / res_chan) and nothing else
    bool fixed_shape = false;  // ber_tconv2.cuh HS: the switches of one shape class as constants (ber_host.cu: tconv2_fixed_shape)
    bool fp64, verify;
    BerSmem (*layout)(int S, int stride, int tail_tx, int tail_rx, int L, int chunk, int use_global);
    const void* fn;
    cudaError_t (*launch)(const BerParams& prm, int grid, size_t smem, cudaStream_t st);
};

template <typename T, int N, int NT, int TC, int LB, int MINB, bool FULL, bool V, int CL = 1, bool CIRC = false, bool TXS = false,
          bool RES = false>
struct BerVariantImpl {
    // grid = CTAs (a multiple of CL); CL > 1 launches thread-block clusters of CL CTAs
    static cudaError_t launch(const BerParams& prm, int grid, size_t smem, cudaStream_t st) {
        if constexpr (CL == 1) {
            ber_frame_kernel<T, N, NT, TC, LB, MINB, FULL, V, 1, CIRC, TXS, RES><<<grid, NT, smem, st>>>(prm);
            return cudaGetLastError();
        } else {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            return cudaLaunchKernelEx(&cfg, ber_frame_kernel<T, N, NT, TC, LB, MINB, FULL, V, CL, CIRC, TXS, RES>, prm);
        }
    }
    static BerVariant make(const char* name) {
        BerVariant v;
        v.name = name; v.N = N; v.NT = NT; v.TC = TC; v.LB = LB; v.MINB = MINB; v.CL = CL; v.circ = CIRC; v.txs = TXS || TC == 0; v.full = FULL; v.ntile = 0; v.gen = 0; v.launch_threads = NT;
        v.fp64 = sizeof(T) == 8; v.verify = V; v.res = RES;
        v.layout = &ber_smem_layout<T, N, NT, TC, LB, RES>;
        v.fn = reinterpret_cast<const void*>(&ber_frame_kernel<T, N, NT, TC, LB, MINB, FULL, V, CL, CIRC, TXS, RES>);
        v.launch = &launch;
        return v;
    }
};

#define WOFDM_VARIANT(T, N, NT, TC, LB, MINB, FULL, tag)                                            \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, false>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL)); \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, true>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_verify"));

// CL CTAs per frame (thread-block cluster)
#define WOFDM_VARIANT_CL(T, N, NT, TC, LB, MINB, FULL, CL, tag)                                     \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, false, CL>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_cl" #CL)); \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, true, CL>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_cl" #CL "_verify"));

// circular-interior policy (one CTA per frame)
#define WOFDM_VARIANT_CIRC(T, N, NT, TC, LB, MINB, FULL, tag)                                       \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, false, 1, true>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_circ")); \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, true, 1, true>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_circ_verify"));

// register-resident kernels that can read the Tx stream from HBM (channel-mask variant); production only
#define WOFDM_VARIANT_TXS(T, N, NT, TC, LB, MINB, FULL, tag)                                        \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, false, 1, false, true>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_txs"));

// kernels with resolved counters (wofdm_ber_run_resolved), production only: the staged policy, and the twins of the register
// policies (CL CTAs per frame, CIRC = circular interior)
#define WOFDM_VARIANT_RES(T, N, NT, tag)                                                                \
    out.push_back(BerVariantImpl<T, N, NT, 0, 0, 1, false, false, 1, false, false, true>::make("ber_" tag "_n" #N "_t" #NT "_c0_l0_b1_f0_res"));
#define WOFDM_VARIANT_RES_REGS(T, N, NT, TC, LB, MINB, FULL, CL, CIRC, tag, sfx)                         \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, false, CL, CIRC, false, true>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_cl" #CL sfx));
// ... and the twins of the TXS instantiations (wofdm_ber_run_masked_resolved: the masked Tx stream read from HBM)
#define WOFDM_VARIANT_RES_TXS(T, N, NT, TC, LB, MINB, FULL, tag)                                         \
    out.push_back(BerVariantImpl<T, N, NT, TC, LB, MINB, FULL, false, 1, false, true, true>::make("ber_" tag "_n" #N "_t" #NT "_c" #TC "_l" #LB "_b" #MINB "_f" #FULL "_txs_res"));

void register_ber_f32_staged(std::vector<BerVariant>& out);
void register_ber_f32_tconv(std::vector<BerVariant>& out);
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
