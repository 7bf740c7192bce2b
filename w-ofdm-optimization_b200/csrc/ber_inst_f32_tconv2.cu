// fp32 instantiations of K1, second generation of the tensor-core-convolution kernel (ber_tconv2.cuh): N = 256, one CTA
// of 256 threads per frame, two CTAs per SM; N = 512, one CTA of 512 threads per frame and SM; NTILE = tiles of 512 stream
// samples (tensor-memory accumulators) per frame.
#include "ber_tconv2_registry.h"
namespace wofdm {
void register_ber_f32_tconv2(std::vector<BerVariant>& out) {
    // channel-mask chain: the Tx stream gathered from the mask product's output (BerParams::tx_y, tconv2_load_masked)
    WOFDM_TCONV2_VARIANT("_txy", 256, 256, 9, 2, false, 1, TCV_LB, true)
    WOFDM_TCONV2_VARIANT("_txy", 256, 256, 10, 2, false, 1, TCV_LB, true)
    WOFDM_TCONV2_VARIANT("_txy", 512, 512, 18, 1, false, 1, TCV_LB, true)
    WOFDM_TCONV2_VARIANT("_txy", 512, 512, 19, 1, false, 1, TCV_LB, true)
    WOFDM_TCONV2_VARIANT("", 256, 256, 9, 2, false)
    WOFDM_TCONV2_VARIANT("_verify", 256, 256, 9, 2, true)
    WOFDM_TCONV2_VARIANT("", 256, 256, 10, 2, false)
    WOFDM_TCONV2_VARIANT("_verify", 256, 256, 10, 2, true)
    WOFDM_TCONV2_VARIANT("", 512, 512, 18, 1, false)
    WOFDM_TCONV2_VARIANT("_verify", 512, 512, 18, 1, true)
    WOFDM_TCONV2_VARIANT("", 512, 512, 19, 1, false)
    WOFDM_TCONV2_VARIANT("_verify", 512, 512, 19, 1, true)
    // N = 1024: a cluster of two CTAs of 512 threads per frame, 8 OFDM symbols and 17..19 tiles per CTA, one CTA per SM
    WOFDM_TCONV2_VARIANT("_cl2", 1024, 512, 18, 1, false, 2)
    WOFDM_TCONV2_VARIANT("_cl2_verify", 1024, 512, 18, 1, true, 2)
    WOFDM_TCONV2_VARIANT("_cl2", 1024, 512, 19, 1, false, 2)
    WOFDM_TCONV2_VARIANT("_cl2_verify", 1024, 512, 19, 1, true, 2)
    // up to 84 taps (BASELINE configs[4]: "L = 21, optionally 84"), N = 256 and the N = 1024 cluster kernel: LB taps of
    // convolution history in the Hankel operand (22 MMAs per tile at LB = 84 instead of 6)
    WOFDM_TCONV2_VARIANT("_cl1_l84", 256, 256, 9, 2, false, 1, 84)
    WOFDM_TCONV2_VARIANT("_cl1_l84_verify", 256, 256, 9, 2, true, 1, 84)
    WOFDM_TCONV2_VARIANT("_cl1_l84", 256, 256, 10, 2, false, 1, 84)
    WOFDM_TCONV2_VARIANT("_cl1_l84_verify", 256, 256, 10, 2, true, 1, 84)
    WOFDM_TCONV2_VARIANT("_cl2_l84", 1024, 512, 18, 1, false, 2, 84)
    WOFDM_TCONV2_VARIANT("_cl2_l84_verify", 1024, 512, 18, 1, true, 2, 84)
    WOFDM_TCONV2_VARIANT("_cl2_l84", 1024, 512, 19, 1, false, 2, 84)
    WOFDM_TCONV2_VARIANT("_cl2_l84_verify", 1024, 512, 19, 1, true, 2, 84)
    // (measured and not kept: the same frames on clusters of 256-thread CTAs, two CTAs of different frames per SM --
    //  N = 512 as 2 x 256 threads: 1.98e8 OFDM symbols/s against 2.06e8; N = 1024 as 4 x 256: 5.5e7 against 8.4e7)
}
}  // namespace wofdm
