// fp32 instantiations of K1, second generation of the tensor-core-convolution kernel (ber_tconv2.cuh): N = 256, one CTA
// of 256 threads per frame, two CTAs per SM; N = 512, one CTA of 512 threads per frame and SM; NTILE = tiles of 512 stream
// samples (tensor-memory accumulators) per frame.
#include "ber_tconv2_registry.h"
namespace wofdm {
#define WOFDM_VARIANT_TCONV2(N, NT, NTILE, MINB)                                                              \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB)); \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, true>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_verify"));
// CL CTAs per frame (thread-block cluster): NTILE tiles per CTA
#define WOFDM_VARIANT_TCONV2_CL(N, NT, NTILE, MINB, CL)                                                       \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false, CL>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_cl" #CL)); \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, true, CL>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_cl" #CL "_verify"));
// long channels: LB taps of convolution history in the Hankel operand (22 MMAs per tile at LB = 84 instead of 6)
#define WOFDM_VARIANT_TCONV2_LB(N, NT, NTILE, MINB, CL, LB)                                                   \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false, CL, LB>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_cl" #CL "_l" #LB)); \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, true, CL, LB>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_cl" #CL "_l" #LB "_verify"));
// channel-mask chain: the Tx stream gathered from the mask product's output (BerParams::tx_y, tconv2_load_masked)
#define WOFDM_VARIANT_TCONV2_TXY(N, NT, NTILE, MINB)                                                          \
    out.push_back(Tconv2VariantImpl<N, NT, NTILE, MINB, false, 1, TCV_LB, true>::make("ber_f32t2_n" #N "_t" #NT "_tiles" #NTILE "_b" #MINB "_txy"));
void register_ber_f32_tconv2(std::vector<BerVariant>& out) {
    WOFDM_VARIANT_TCONV2_TXY(256, 256, 9, 2)
    WOFDM_VARIANT_TCONV2_TXY(256, 256, 10, 2)
    WOFDM_VARIANT_TCONV2_TXY(512, 512, 18, 1)
    WOFDM_VARIANT_TCONV2_TXY(512, 512, 19, 1)
    WOFDM_VARIANT_TCONV2(256, 256, 9, 2)
    WOFDM_VARIANT_TCONV2(256, 256, 10, 2)
    WOFDM_VARIANT_TCONV2(512, 512, 18, 1)
    WOFDM_VARIANT_TCONV2(512, 512, 19, 1)
    // N = 1024: a cluster of two CTAs of 512 threads per frame, 8 OFDM symbols and 17..19 tiles per CTA, one CTA per SM
    WOFDM_VARIANT_TCONV2_CL(1024, 512, 18, 1, 2)
    WOFDM_VARIANT_TCONV2_CL(1024, 512, 19, 1, 2)
    // up to 84 taps (BASELINE configs[4]: "L = 21, optionally 84"), N = 256 and the N = 1024 cluster kernel
    WOFDM_VARIANT_TCONV2_LB(256, 256, 9, 2, 1, 84)
    WOFDM_VARIANT_TCONV2_LB(256, 256, 10, 2, 1, 84)
    WOFDM_VARIANT_TCONV2_LB(1024, 512, 18, 1, 2, 84)
    WOFDM_VARIANT_TCONV2_LB(1024, 512, 19, 1, 2, 84)
    // (measured and not kept: the same frames on clusters of 256-thread CTAs, two CTAs of different frames per SM --
    //  N = 512 as 2 x 256 threads: 1.98e8 OFDM symbols/s against 2.06e8; N = 1024 as 4 x 256: 5.5e7 against 8.4e7)
}
}  // namespace wofdm
