// fp32 instantiations of the register-resident K1 policy (production path).
// WOFDM_VARIANT(tag, name suffix, type, N, threads, TC = samples per thread, LB = taps in registers (L <= LB), min CTAs/SM,
//               FULL = threads*TC == S*stride exactly, verify instance[, CL, CIRC, TXS, RES])
#include "ber_registry.h"
namespace wofdm {
void register_ber_f32_regs(std::vector<BerVariant>& out) {
    register_ber_f32_regs_big(out);
    WOFDM_VARIANT("f32r", "", float, 256, 256, 17, 21, 2, true, false)
    WOFDM_VARIANT("f32r", "_verify", float, 256, 256, 17, 21, 2, true, true)
    WOFDM_VARIANT("f32r", "", float, 256, 256, 17, 21, 2, false, false)
    WOFDM_VARIANT("f32r", "_verify", float, 256, 256, 17, 21, 2, false, true)
    WOFDM_VARIANT("f32r", "", float, 256, 256, 19, 21, 2, false, false)
    WOFDM_VARIANT("f32r", "_verify", float, 256, 256, 19, 21, 2, false, true)
    WOFDM_VARIANT("f32r", "_circ", float, 256, 256, 17, 21, 2, true, false, 1, true)
    WOFDM_VARIANT("f32r", "_circ_verify", float, 256, 256, 17, 21, 2, true, true, 1, true)
    WOFDM_VARIANT("f32r", "_circ", float, 256, 256, 17, 21, 2, false, false, 1, true)
    WOFDM_VARIANT("f32r", "_circ_verify", float, 256, 256, 17, 21, 2, false, true, 1, true)
    WOFDM_VARIANT("f32r", "_circ", float, 256, 256, 19, 21, 2, false, false, 1, true)
    WOFDM_VARIANT("f32r", "_circ_verify", float, 256, 256, 19, 21, 2, false, true, 1, true)
}
}  // namespace wofdm
