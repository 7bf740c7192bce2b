// fp32 instantiations of the register-resident K1 policy for N = 512 and N = 1024 (own translation unit: build time).
#include "ber_registry.h"
namespace wofdm {
void register_ber_f32_regs_big(std::vector<BerVariant>& out) {
    // N = 256 with the Tx stream taken from HBM (channel-mask variant, matlab/main_channel_mask.m)
    WOFDM_VARIANT("f32r", "_txs", float, 256, 256, 17, 21, 2, true, false, 1, false, true)
    WOFDM_VARIANT("f32r", "_txs", float, 256, 256, 17, 21, 2, false, false, 1, false, true)
    WOFDM_VARIANT("f32r", "_txs", float, 256, 256, 19, 21, 2, false, false, 1, false, true)
    // N = 512: one CTA of 512 threads per frame (one per SM: stream + parked noise = 140 KB)
    WOFDM_VARIANT("f32r", "", float, 512, 512, 17, 21, 1, true, false)
    WOFDM_VARIANT("f32r", "_verify", float, 512, 512, 17, 21, 1, true, true)
    WOFDM_VARIANT("f32r", "", float, 512, 512, 17, 21, 1, false, false)
    WOFDM_VARIANT("f32r", "_verify", float, 512, 512, 17, 21, 1, false, true)
    WOFDM_VARIANT("f32r", "", float, 512, 512, 19, 21, 1, false, false)
    WOFDM_VARIANT("f32r", "_verify", float, 512, 512, 19, 21, 1, false, true)
    // N = 1024: one frame per 2-CTA cluster, 8 OFDM symbols and 512 threads per CTA (ber_kernel.cuh, CL)
    WOFDM_VARIANT("f32r", "_cl2", float, 1024, 512, 17, 21, 1, true, false, 2)
    WOFDM_VARIANT("f32r", "_cl2_verify", float, 1024, 512, 17, 21, 1, true, true, 2)
    WOFDM_VARIANT("f32r", "_cl2", float, 1024, 512, 17, 21, 1, false, false, 2)
    WOFDM_VARIANT("f32r", "_cl2_verify", float, 1024, 512, 17, 21, 1, false, true, 2)
    WOFDM_VARIANT("f32r", "_cl2", float, 1024, 512, 19, 21, 1, false, false, 2)
    WOFDM_VARIANT("f32r", "_cl2_verify", float, 1024, 512, 19, 21, 1, false, true, 2)
}
}  // namespace wofdm
