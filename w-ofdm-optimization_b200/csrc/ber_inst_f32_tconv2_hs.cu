// The production tensor-core K1 kernels at N = 256 (ber_inst_f32_tconv2.cu) with the frame loop compiled for the common
// shape class (ber_tconv2.cuh: HS): flat Tx window, no Rx tails, one window pair, no guard band, symbols drawn in the kernel.
// A translation unit of its own, so that the generic kernels keep their code.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_hs(std::vector<BerVariant>& out) {
    WOFDM_TCONV2_VARIANT("_hs", 256, 256, 9, 2, false, 1, TCV_LB, false, false, true)
    WOFDM_TCONV2_VARIANT("_hs", 256, 256, 10, 2, false, 1, TCV_LB, false, false, true)
}
}  // namespace wofdm
