// Resolved-counter twins (RES) of the staged K1 policy, fp32 and fp64 (ber_inst_f32_staged.cu, ber_inst_f64_staged.cu).
#include "ber_registry.h"
namespace wofdm {
void register_ber_staged_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT_RES(float, 16, 32, "f32")
    WOFDM_VARIANT_RES(float, 32, 32, "f32")
    WOFDM_VARIANT_RES(float, 64, 64, "f32")
    WOFDM_VARIANT_RES(float, 128, 128, "f32")
    WOFDM_VARIANT_RES(float, 256, 256, "f32")
    WOFDM_VARIANT_RES(float, 512, 256, "f32")
    WOFDM_VARIANT_RES(float, 1024, 512, "f32")
    WOFDM_VARIANT_RES(double, 16, 32, "f64")
    WOFDM_VARIANT_RES(double, 32, 32, "f64")
    WOFDM_VARIANT_RES(double, 64, 64, "f64")
    WOFDM_VARIANT_RES(double, 128, 128, "f64")
    WOFDM_VARIANT_RES(double, 256, 256, "f64")
    WOFDM_VARIANT_RES(double, 512, 256, "f64")
    WOFDM_VARIANT_RES(double, 1024, 256, "f64")
}
}  // namespace wofdm
