// fp64 instantiations of the staged K1 policy (verify-grade arithmetic).
#include "ber_registry.h"
namespace wofdm {
void register_ber_f64_staged(std::vector<BerVariant>& out) {
    WOFDM_VARIANT("f64", "", double, 16, 32, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 16, 32, 0, 0, 1, false, true)
    WOFDM_VARIANT("f64", "", double, 32, 32, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 32, 32, 0, 0, 1, false, true)
    WOFDM_VARIANT("f64", "", double, 64, 64, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 64, 64, 0, 0, 1, false, true)
    WOFDM_VARIANT("f64", "", double, 128, 128, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 128, 128, 0, 0, 1, false, true)
    WOFDM_VARIANT("f64", "", double, 256, 256, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 256, 256, 0, 0, 1, false, true)
    WOFDM_VARIANT("f64", "", double, 512, 256, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 512, 256, 0, 0, 1, false, true)
    WOFDM_VARIANT("f64", "", double, 1024, 256, 0, 0, 1, false, false)
    WOFDM_VARIANT("f64", "_verify", double, 1024, 256, 0, 0, 1, false, true)
}
}  // namespace wofdm
