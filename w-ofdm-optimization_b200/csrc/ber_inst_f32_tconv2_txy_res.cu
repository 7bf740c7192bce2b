// Resolved-counter twins (RES) of the channel-mask chain's tensor-core K1 kernels that gather the Tx stream from the mask
// product (TXY, ber_inst_f32_tconv2.cu).  Own translation unit, so that every production object keeps its code.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_txy_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT_TCONV2_TXY_RES(256, 256, 9, 2)
    WOFDM_VARIANT_TCONV2_TXY_RES(256, 256, 10, 2)
    WOFDM_VARIANT_TCONV2_TXY_RES(512, 512, 18, 1)
    WOFDM_VARIANT_TCONV2_TXY_RES(512, 512, 19, 1)
}
}  // namespace wofdm
