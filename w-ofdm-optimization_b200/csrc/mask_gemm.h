// mask_gemm.h -- the channel-mask Tx chain as one dense tensor-core product (mask_gemm.cu), used by wofdm_ber_run_masked.
#pragma once
#include <cuda_fp16.h>
#include "host_common.h"

namespace wofdm {

// n_var mask matrices (window pairs) over one B operand.  Device footprint per pair at N = 256 (n_tx = 280, Yp = 640) and
// the channel-mask chain's batch of 16 384 frames of S = 16: Y 0.67 GB, A 1 MB; shared by all pairs: B 0.27 GB.
struct MaskGemm {
    int N, S, n_tx, stride, tail_tx, cp, bits, guard;
    int nvar;           // window pairs: pair v's [Mtop | Mbot] is row tiles [v RT, (v+1) RT) of A, its output Y + v ypair
    int M;              // 2 n_tx - 1: length of the mask's circular convolution
    int nact;           // active sub-carriers N - 2 guard
    int Kp, nk;         // K = 2 halves of 2 nact (Re, Im interleaved; symbols s and s-1), each rounded up to the K block; K blocks
    int RT, Yp;         // row tiles of 128 per pair; floats per column of Y (= RT * 128 >= 2 n_tx)
    long long batch;    // frames per batch (columns = batch * S, rounded up to the column tile)
    long long ypair;    // floats between two pairs' outputs (columns * Yp)
    __half* At;         // mask matrices, [nvar][RT][nk][hi | lo][128 x 64] K-major UMMA tiles
    __half* Bt;         // lattice points of the batch's symbols, [CT][nk][256 x 64] tiles
    float* Y;           // [nvar][columns][Yp]: pair v's filtered symbol of column (frame, s) -- its n_tx samples with the filter
                        // tail of symbol s-1 added -- (Re, Im) interleaved
    float* scale;       // [nvar][2]: power-of-two scale of pair v's A and its inverse (set on the device)
    double2* g;         // [M] impulse response of the mask (of the pair being set up)
    double2* Mm;        // [M][nact] the matrix in fp64 before the split (of the pair being set up)
    unsigned* maxbits;  // [nvar] largest |entry| of pair v's matrix as float bits
};

// dimensions for `sys`, `batch` frames and nvar window pairs; returns the device bytes mask_gemm_setup takes from the arena
size_t mask_gemm_plan(const wofdm_sys_t& sys, long long batch, int nvar, MaskGemm& mg);
// arena buffers + the matrices: pair v's mask of roll_off[v] bins (main_channel_mask.m:404-412, 477-493) on its Tx table
// d_wtx + v n_tx (K1's tables, back to back).  roll_off[v] == 0: g = delta instead of the mask, so Mtop = the windowed,
// CP-extended IDFT columns and Mbot = 0 -- the UNMASKED symbols through the same product (wofdm_psd_masked's unmasked
// spectra; the BER chain's roll-offs are all >= 1)
int mask_gemm_setup(wofdm_ctx* h, DeviceCtx& d, MaskGemm& mg, const int* roll_off, const float* d_wtx);
// masked symbols of frames f0 .. f0 + nf - 1 (nf <= batch) of every pair into Y: the symbols are drawn once, one product
// covers all pairs.  seg (a device segment table [n_seg][4], BerParams::seg): f0 .. f0 + nf - 1 are local indices of the
// segment list of a job with C channels and `ensemble` ensemble indices per point
int mask_gemm_batch(wofdm_ctx* h, DeviceCtx& d, const MaskGemm& mg, uint64_t seed, long long f0, long long nf,
                    const long long* seg = nullptr, int n_seg = 0, int C = 0, long long ensemble = 0);
// pair v's serialised Tx streams of the last batch's nf frames, from Y, into stream[nf][tail_tx + S * stride]
int mask_gemm_assemble(wofdm_ctx* h, DeviceCtx& d, const MaskGemm& mg, int v, long long nf, float2* stream);

}  // namespace wofdm
