// Resolved-counter twins (RES) of the register-resident K1 kernels (ber_inst_f32_regs.cu, ber_inst_f32_regs_big.cu): the same
// arithmetic and noise blocks as the kernel production picks, so the resolved counters add up to its counters bit for bit.
#include "ber_registry.h"
namespace wofdm {
void register_ber_f32_regs_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT_RES_REGS(float, 256, 256, 17, 21, 2, true, 1, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 256, 256, 17, 21, 2, false, 1, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 256, 256, 19, 21, 2, false, 1, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 256, 256, 17, 21, 2, true, 1, true, "f32r", "_circ_res")
    WOFDM_VARIANT_RES_REGS(float, 256, 256, 17, 21, 2, false, 1, true, "f32r", "_circ_res")
    WOFDM_VARIANT_RES_REGS(float, 256, 256, 19, 21, 2, false, 1, true, "f32r", "_circ_res")
    WOFDM_VARIANT_RES_REGS(float, 512, 512, 17, 21, 1, true, 1, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 512, 512, 17, 21, 1, false, 1, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 512, 512, 19, 21, 1, false, 1, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 1024, 512, 17, 21, 1, true, 2, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 1024, 512, 17, 21, 1, false, 2, false, "f32r", "_res")
    WOFDM_VARIANT_RES_REGS(float, 1024, 512, 19, 21, 1, false, 2, false, "f32r", "_res")
}
}  // namespace wofdm
