// The production tensor-core K1 kernels at N = 256 (ber_inst_f32_tconv2.cu) with the frame loop compiled for the common
// shape class (ber_tconv2.cuh: HS): flat Tx window, no Rx tails, one window pair, no guard band, symbols drawn in the kernel.
// "_hs": the geometry of bench.py's headline compiled in as well (TCV2_HS_WTX256; a headline frame needs 9 tiles under
// either noise normalisation); "_hsc": the class with its geometry at run time, for every other shape of the class.
// A translation unit of its own, so that the generic kernels keep their code.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2_hs(std::vector<BerVariant>& out) {
    WOFDM_TCONV2_VARIANT("_hs", 256, 256, 9, 2, false, 1, TCV_LB, false, false, TCV2_HS_WTX256)
    WOFDM_TCONV2_VARIANT("_hsc", 256, 256, 9, 2, false, 1, TCV_LB, false, false, TCV2_HS_CLASS)
    WOFDM_TCONV2_VARIANT("_hsc", 256, 256, 10, 2, false, 1, TCV_LB, false, false, TCV2_HS_CLASS)
}
}  // namespace wofdm
