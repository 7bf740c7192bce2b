// fp32 instantiations of the staged (fully general) K1 policy.
#include "ber_registry.h"
namespace wofdm {
void register_ber_f32_staged(std::vector<BerVariant>& out) {
    WOFDM_VARIANT("f32", "", float, 16, 32, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 16, 32, 0, 0, 1, false, true)
    WOFDM_VARIANT("f32", "", float, 32, 32, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 32, 32, 0, 0, 1, false, true)
    WOFDM_VARIANT("f32", "", float, 64, 64, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 64, 64, 0, 0, 1, false, true)
    WOFDM_VARIANT("f32", "", float, 128, 128, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 128, 128, 0, 0, 1, false, true)
    WOFDM_VARIANT("f32", "", float, 256, 256, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 256, 256, 0, 0, 1, false, true)
    WOFDM_VARIANT("f32", "", float, 512, 256, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 512, 256, 0, 0, 1, false, true)
    WOFDM_VARIANT("f32", "", float, 1024, 512, 0, 0, 1, false, false)
    WOFDM_VARIANT("f32", "_verify", float, 1024, 512, 0, 0, 1, false, true)
}
}  // namespace wofdm
