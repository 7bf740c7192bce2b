// Resolved-counter twins (RES) of the production tensor-core K1 kernels (ber_inst_f32_tconv2.cu): the N = 1024 two-CTA
// cluster and the LB = 84 long-channel instances.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_res_big(std::vector<BerVariant>& out) {
    WOFDM_TCONV2_VARIANT("_cl2_lTCV_LB_res", 1024, 512, 18, 1, false, 2, TCV_LB, false, true)
    WOFDM_TCONV2_VARIANT("_cl2_lTCV_LB_res", 1024, 512, 19, 1, false, 2, TCV_LB, false, true)
    WOFDM_TCONV2_VARIANT("_cl1_l84_res", 256, 256, 9, 2, false, 1, 84, false, true)
    WOFDM_TCONV2_VARIANT("_cl1_l84_res", 256, 256, 10, 2, false, 1, 84, false, true)
    WOFDM_TCONV2_VARIANT("_cl2_l84_res", 1024, 512, 18, 1, false, 2, 84, false, true)
    WOFDM_TCONV2_VARIANT("_cl2_l84_res", 1024, 512, 19, 1, false, 2, 84, false, true)
}
}  // namespace wofdm
