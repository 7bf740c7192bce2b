// Resolved-counter twins (RES) of the production tensor-core K1 kernels (ber_inst_f32_tconv2.cu): N = 256 and 512, one CTA
// per frame.  Separate instantiations, so that the production kernels keep their code.  (The names of the LB = TCV_LB twins
// spell "TCV_LB", as they always have.)
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_res(std::vector<BerVariant>& out) {
    WOFDM_TCONV2_VARIANT("_cl1_lTCV_LB_res", 256, 256, 9, 2, false, 1, TCV_LB, false, true)
    WOFDM_TCONV2_VARIANT("_cl1_lTCV_LB_res", 256, 256, 10, 2, false, 1, TCV_LB, false, true)
    WOFDM_TCONV2_VARIANT("_cl1_lTCV_LB_res", 512, 512, 18, 1, false, 1, TCV_LB, false, true)
    WOFDM_TCONV2_VARIANT("_cl1_lTCV_LB_res", 512, 512, 19, 1, false, 1, TCV_LB, false, true)
    register_ber_f32_tconv2_res_big(out);
}
}  // namespace wofdm
