// Resolved-counter twins (RES) of the register-resident K1 kernels (ber_inst_f32_regs.cu, ber_inst_f32_regs_big.cu): the same
// arithmetic and noise blocks as the kernel production picks, so the resolved counters add up to its counters bit for bit.
#include "ber_registry.h"
namespace wofdm {
void register_ber_f32_regs_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT("f32r", "_cl1_res", float, 256, 256, 17, 21, 2, true, false, 1, false, false, true)
    WOFDM_VARIANT("f32r", "_cl1_res", float, 256, 256, 17, 21, 2, false, false, 1, false, false, true)
    WOFDM_VARIANT("f32r", "_cl1_res", float, 256, 256, 19, 21, 2, false, false, 1, false, false, true)
    WOFDM_VARIANT("f32r", "_cl1_circ_res", float, 256, 256, 17, 21, 2, true, false, 1, true, false, true)
    WOFDM_VARIANT("f32r", "_cl1_circ_res", float, 256, 256, 17, 21, 2, false, false, 1, true, false, true)
    WOFDM_VARIANT("f32r", "_cl1_circ_res", float, 256, 256, 19, 21, 2, false, false, 1, true, false, true)
    WOFDM_VARIANT("f32r", "_cl1_res", float, 512, 512, 17, 21, 1, true, false, 1, false, false, true)
    WOFDM_VARIANT("f32r", "_cl1_res", float, 512, 512, 17, 21, 1, false, false, 1, false, false, true)
    WOFDM_VARIANT("f32r", "_cl1_res", float, 512, 512, 19, 21, 1, false, false, 1, false, false, true)
    WOFDM_VARIANT("f32r", "_cl2_res", float, 1024, 512, 17, 21, 1, true, false, 2, false, false, true)
    WOFDM_VARIANT("f32r", "_cl2_res", float, 1024, 512, 17, 21, 1, false, false, 2, false, false, true)
    WOFDM_VARIANT("f32r", "_cl2_res", float, 1024, 512, 19, 21, 1, false, false, 2, false, false, true)
}
}  // namespace wofdm
