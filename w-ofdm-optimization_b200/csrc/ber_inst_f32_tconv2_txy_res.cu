// Resolved-counter twins (RES) of the channel-mask chain's tensor-core K1 kernels that gather the Tx stream from the mask
// product (TXY, ber_inst_f32_tconv2.cu).  Own translation unit, so that every production object keeps its code.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_txy_res(std::vector<BerVariant>& out) {
    WOFDM_TCONV2_VARIANT("_txy_res", 256, 256, 9, 2, false, 1, TCV_LB, true, true)
    WOFDM_TCONV2_VARIANT("_txy_res", 256, 256, 10, 2, false, 1, TCV_LB, true, true)
    WOFDM_TCONV2_VARIANT("_txy_res", 512, 512, 18, 1, false, 1, TCV_LB, true, true)
    WOFDM_TCONV2_VARIANT("_txy_res", 512, 512, 19, 1, false, 1, TCV_LB, true, true)
}
}  // namespace wofdm
