// mask_gemm.h -- the channel-mask Tx chain as one dense tensor-core product (mask_gemm.cu), used by wofdm_ber_run_masked.
#pragma once
#include <cuda_fp16.h>
#include "host_common.h"

namespace wofdm {

struct MaskGemm {
    int N, S, n_tx, stride, tail_tx, cp, bits, guard;
    int M;              // 2 n_tx - 1: length of the mask's circular convolution
    int nact;           // active sub-carriers N - 2 guard
    int Kp, nk;         // K = 2 halves of 2 nact (Re, Im interleaved; symbols s and s-1), each rounded up to the K block; K blocks
    int RT, Yp;         // row tiles of 128; floats per column of Y (= RT * 128 >= 2 n_tx)
    long long batch;    // frames per batch (columns = batch * S, rounded up to the column tile)
    __half* At;         // mask matrix, [RT][nk][hi | lo][128 x 64] K-major UMMA tiles
    __half* Bt;         // lattice points of the batch's symbols, [CT][nk][256 x 64] tiles
    float* Y;           // [columns][Yp]: the filtered symbol of column (frame, s) -- its n_tx samples with the filter tail of symbol
                        // s-1 added -- (Re, Im) interleaved
    float* scale;       // [2]: power-of-two scale of At and its inverse (set on the device)
    double2* g;         // [M] impulse response of the mask
    double2* Mm;        // [M][nact] the matrix in fp64 before the split
    unsigned* maxbits;  // largest |entry| as float bits
};

// dimensions for `sys` and `batch` frames; returns the device bytes mask_gemm_setup takes from the arena
size_t mask_gemm_plan(const wofdm_sys_t& sys, long long batch, MaskGemm& mg);
// arena buffers + the matrix: the mask of roll_off bins (main_channel_mask.m:404-412, 477-493), d_wtx = K1's Tx table
int mask_gemm_setup(wofdm_ctx* h, DeviceCtx& d, MaskGemm& mg, int roll_off, const float* d_wtx);
// masked symbols of frames f0 .. f0 + nf - 1 (nf <= batch) into Y and, if `stream` is not NULL, the serialised Tx streams
// into stream[nf][tail_tx + S * stride].  seg (a device segment table [n_seg][4], BerParams::seg): f0 .. f0 + nf - 1 are
// local indices of the segment list of a job with C channels and `ensemble` ensemble indices per point
int mask_gemm_batch(wofdm_ctx* h, DeviceCtx& d, const MaskGemm& mg, uint64_t seed, long long f0, long long nf, float2* stream,
                    const long long* seg = nullptr, int n_seg = 0, int C = 0, long long ensemble = 0);

}  // namespace wofdm
