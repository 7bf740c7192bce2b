// Resolved-counter twins (RES) of the channel-mask chain's register-resident K1 kernels that read the assembled Tx stream
// (TXS, ber_inst_f32_regs_big.cu).  Own translation unit, so that every production object keeps its code.
#include "ber_registry.h"
namespace wofdm {
void register_ber_f32_regs_txs_res(std::vector<BerVariant>& out) {
    WOFDM_VARIANT("f32r", "_txs_res", float, 256, 256, 17, 21, 2, true, false, 1, false, true, true)
    WOFDM_VARIANT("f32r", "_txs_res", float, 256, 256, 17, 21, 2, false, false, 1, false, true, true)
    WOFDM_VARIANT("f32r", "_txs_res", float, 256, 256, 19, 21, 2, false, false, 1, false, true, true)
}
}  // namespace wofdm
