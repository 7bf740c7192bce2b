// Resolved-counter twins (RES) of the production tensor-core K1 kernels (ber_inst_f32_tconv2.cu): the N = 1024 two-CTA
// cluster and the LB = 84 long-channel instances.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_res_big(std::vector<BerVariant>& out) {
    WOFDM_VARIANT_TCONV2_RES(1024, 512, 18, 1, 2, TCV_LB)
    WOFDM_VARIANT_TCONV2_RES(1024, 512, 19, 1, 2, TCV_LB)
    WOFDM_VARIANT_TCONV2_RES(256, 256, 9, 2, 1, 84)
    WOFDM_VARIANT_TCONV2_RES(256, 256, 10, 2, 1, 84)
    WOFDM_VARIANT_TCONV2_RES(1024, 512, 18, 1, 2, 84)
    WOFDM_VARIANT_TCONV2_RES(1024, 512, 19, 1, 2, 84)
}
}  // namespace wofdm
