// ber_tconv2_registry.h -- registry entries of the second-generation tensor-core K1 kernel (ber_tconv2.cuh).
#pragma once
#include "ber_registry.h"
#include "ber_tconv2.cuh"
namespace wofdm {
template <int N, int NT, int NTILE, int MINB, bool V, int CL = 1, int LB = TCV_LB, bool TXY = false, bool RES = false,
          bool HS = false>
struct Tconv2VariantImpl {
    // grid = CTAs (a multiple of CL); CL > 1 launches thread-block clusters of CL CTAs
    static cudaError_t launch(const BerParams& prm, int grid, size_t smem, cudaStream_t st) {
        if constexpr (CL == 1) {
            ber_tconv2_kernel<N, NT, NTILE, MINB, V, 1, LB, TXY, RES, HS><<<grid, NT + tconv2_mma_warp_threads(N, NT), smem, st>>>(prm);   // (+ the MMA warp)
            return cudaGetLastError();
        } else {
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NT + tconv2_mma_warp_threads(N, NT)); cfg.dynamicSmemBytes = smem; cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            return cudaLaunchKernelEx(&cfg, ber_tconv2_kernel<N, NT, NTILE, MINB, V, CL, LB, TXY, RES, HS>, prm);
        }
    }
    static BerVariant make(const char* name) {
        BerVariant v;
        v.name = name; v.N = N; v.NT = NT; v.TC = 2 * NTILE; v.LB = LB; v.MINB = MINB; v.CL = CL; v.circ = false; v.txs = !HS; v.full = false;
        v.ntile = NTILE; v.gen = 2; v.txy = TXY; v.res = RES; v.fixed_shape = HS; v.launch_threads = NT + tconv2_mma_warp_threads(N, NT);
        v.fp64 = false; v.verify = V;
        // (txs = !HS is descriptive only: choose_variant compares txs on the register policies, and keeps HS off the Tx-stream
        //  path through tconv2_fixed_shape(!want_txs))
        v.layout = &tconv2_smem_layout<N, NT, NTILE, LB, RES>;
        v.fn = reinterpret_cast<const void*>(&ber_tconv2_kernel<N, NT, NTILE, MINB, V, CL, LB, TXY, RES, HS>);
        v.launch = &launch;
        return v;
    }
};
// counters resolved by sub-carrier / channel (wofdm_ber_run_resolved): the production kernels' twins, registered separately
#define WOFDM_VARIANT_TCONV2_RES(N, NT, NTILE, MINB, CL, LB)                                                  \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false, CL, LB, false, true>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_cl" #CL "_l" #LB "_res"));
// the twins of the TXY instantiations (wofdm_ber_run_masked_resolved: the Tx stream gathered from the mask product)
#define WOFDM_VARIANT_TCONV2_TXY_RES(N, NT, NTILE, MINB)                                                      \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false, 1, TCV_LB, true, true>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_txy_res"));
// the fixed-shape frame loop of the production kernels (ber_tconv2.cuh: HS; ber_host.cu: tconv2_fixed_shape)
#define WOFDM_VARIANT_TCONV2_HS(N, NT, NTILE, MINB)                                                           \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false, 1, TCV_LB, false, false, true>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_hs"));
}  // namespace wofdm
