// Resolved-counter twins (RES) of the staged K1 policy, fp32 and fp64 (ber_inst_f32_staged.cu, ber_inst_f64_staged.cu).
#include "ber_registry.h"
namespace wofdm {
void register_ber_staged_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT("f32", "_res", float, 16, 32, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f32", "_res", float, 32, 32, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f32", "_res", float, 64, 64, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f32", "_res", float, 128, 128, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f32", "_res", float, 256, 256, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f32", "_res", float, 512, 256, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f32", "_res", float, 1024, 512, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 16, 32, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 32, 32, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 64, 64, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 128, 128, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 256, 256, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 512, 256, 0, 0, 1, 0, false, 1, false, false, true)
    WOFDM_VARIANT("f64", "_res", double, 1024, 256, 0, 0, 1, 0, false, 1, false, false, true)
}
}  // namespace wofdm
