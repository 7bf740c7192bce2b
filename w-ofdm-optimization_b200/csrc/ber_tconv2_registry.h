// ber_tconv2_registry.h -- registry entries of the second-generation tensor-core K1 kernel (ber_tconv2.cuh).
#pragma once
#include "ber_registry.h"
#include "ber_tconv2.cuh"
namespace wofdm {
template <int N, int NT, int NTILE, int MINB, bool V, int CL = 1, int LB = TCV_LB, bool TXY = false, bool RES = false,
          int HS = 0>
struct Tconv2VariantImpl {
    static BerVariant make(const char* name) {
        constexpr auto kernel = &ber_tconv2_kernel<N, NT, NTILE, MINB, V, CL, LB, TXY, RES, HS>;
        BerVariant v;
        v.name = name; v.N = N; v.NT = NT; v.TC = 2 * NTILE; v.LB = LB; v.MINB = MINB; v.CL = CL; v.circ = false; v.full = false;
        v.ntile = NTILE; v.txy = TXY; v.res = RES; v.fixed_shape = HS != 0; v.geom = tconv2_geom(HS).N > 0 ? HS : 0; v.launch_threads = NT + tconv2_mma_warp_threads(N, NT);   // (+ the MMA warp)
        v.fp64 = false; v.verify = V;
        v.layout = &tconv2_smem_layout<N, NT, NTILE, LB, RES>;
        v.fn = reinterpret_cast<const void*>(kernel);
        v.launch = &launch_frames<kernel, NT + tconv2_mma_warp_threads(N, NT), CL>;
        return v;
    }
};
// ber_tconv2_kernel<N, NT, NTILE, MINB, ...> registered as "ber_f32t2_n<N>_t<NT>_tiles<NTILE>_b<MINB><sfx>"; "..." are the
// template arguments from V on (V = verify instance, CL, LB, TXY, RES, HS: TCV2_HS_CLASS or a geometry id)
#define WOFDM_TCONV2_VARIANT(sfx, N, NT, NTILE, MINB, ...)                                                    \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, __VA_ARGS__>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB sfx));
}  // namespace wofdm
