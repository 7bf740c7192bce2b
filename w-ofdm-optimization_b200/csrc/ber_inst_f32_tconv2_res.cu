// Resolved-counter twins (RES) of the production tensor-core K1 kernels (ber_inst_f32_tconv2.cu): N = 256 and 512, one CTA
// per frame.  Separate instantiations, so that the production kernels keep their code.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT_TCONV2_RES(256, 256, 9, 2, 1, TCV_LB)
    WOFDM_VARIANT_TCONV2_RES(256, 256, 10, 2, 1, TCV_LB)
    WOFDM_VARIANT_TCONV2_RES(512, 512, 18, 1, 1, TCV_LB)
    WOFDM_VARIANT_TCONV2_RES(512, 512, 19, 1, 1, TCV_LB)
    register_ber_f32_tconv2_res_big(out);
}
}  // namespace wofdm
