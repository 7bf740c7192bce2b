// psd_masked.cu -- PSD of the channel-mask chain's Tx streams, masked and unmasked, on the frames of its BER calls.
//
// The mask product (mask_gemm.cu) writes every filtered symbol of a batch of frames into Y: column (frame, s) holds
// f_s = y_s[0..n_tx) + y_{s-1}[n_tx..M).  A frame's serialised stream is the overlap-add of its columns with the frame
// stride (the rule of mask_assemble_kernel and of the K1 loader tconv2_load_masked):
//     stream[s stride + i] = f_s[i] + f_{s-1}[stride + i]   (the second term while stride + i < n_tx; zero past len)
// psd_masked_kernel reads its slices straight from Y by that rule, so no assembled stream is written.  The unmasked
// stream is the same product with the mask's impulse response replaced by a unit impulse (mask_gemm_setup, roll-off 0):
// every requested spectrum -- masked and unmasked, of every configuration -- is one pair of a single product, so a batch's
// symbols are drawn once and all spectra come from one code path on identical symbols.
//
// Spectrum p is blockIdx.y.  One CTA of 256 threads works on G = 256 / (8N/16) slices of one frame at a time (4 / 2 / 1 for
// N = 128 / 256 / 512):
// each thread loads its 16 samples of its slice, applies the taper (estimator 1), runs the 8N-point register FFT and
// keeps |X|^2 in fp64 registers over all of the CTA's items; one fftshift-indexed atomicAdd(double) per bin and CTA at
// the end, as psd_kernel (psd.cu) does.  fp32 arithmetic, fp64 accumulation.
#include <algorithm>
#include <cstring>

#include "host_common.h"
#include "mask_gemm.h"

namespace wofdm {
namespace {

struct PsdMaskedParams {
    const float* Y;                // [spectra][frames * S][Yp]: the filtered symbols of the batch, (Re, Im) interleaved
    long long ypair;               // floats between two spectra's columns (MaskGemm::ypair)
    int Yp, S, stride, n_tx;
    int len;                       // samples of a frame's stream: tail_tx + S * stride
    int n_slices;                  // slices per frame
    int groups;                    // ceil(n_slices / G)
    int hop;                       // first sample of slice k: k * hop (8N, or 4N for the Hann estimator)
    int hann;                      // taper sin^2(pi n / 8N)
    long long items;               // frames of the batch * groups
    const float2* twp;             // twiddles of the 8N-point transform
    double* psd;                   // [spectra][8N], sum over slices and frames
};

template <int N>
__global__ void __launch_bounds__(256, 2) psd_masked_kernel(const PsdMaskedParams p) {
    constexpr int P = 8 * N;
    using PP = FftPlan<P>;
    constexpr int TPF = PP::TPF, G = 256 / TPF;
    extern __shared__ __align__(16) unsigned char psm[];
    float2* twp = reinterpret_cast<float2*>(psm);
    float2* xb = twp + PP::NTW;                            // G exchange buffers (NTW is even: 16-byte aligned)
    const int tid = threadIdx.x, slot = tid / TPF, t = tid % TPF;
    for (int i = tid; i < PP::NTW; i += 256) twp[i] = p.twp[i];
    float tap[16];                                         // a thread's samples sit at the same offsets in every slice
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const float s = sinpif((float)(t + q * TPF) / (float)P);
        tap[q] = p.hann ? s * s : 1.f;
    }
    __syncthreads();

    double acc[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) acc[q] = 0.0;
    for (long long it = blockIdx.x; it < p.items; it += gridDim.x) {
        const long long fl = it / p.groups;
        const int k = (int)(it - fl * p.groups) * G + slot;
        const bool live = k < p.n_slices;
        const int a0 = k * p.hop;
        const float* yf = p.Y + (size_t)blockIdx.y * p.ypair + (size_t)fl * p.S * p.Yp;
        float2 v[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int pos = a0 + t + q * TPF;
            float2 x = make_float2(0.f, 0.f);
            if (live && pos < p.len) {
                const int s = min(pos / p.stride, p.S), i = pos - s * p.stride;
                const float* ys = yf + (size_t)s * p.Yp;
                if (s < p.S) x = *reinterpret_cast<const float2*>(ys + 2 * i);
                if (s >= 1 && p.stride + i < p.n_tx) x = cadd(x, *reinterpret_cast<const float2*>(ys - p.Yp + 2 * (p.stride + i)));
            }
            v[q] = make_float2(x.x * tap[q], x.y * tap[q]);
        }
        fft_regs<float, P, -1, G>(v, t, xb + slot * PP::XLEN, twp, slot);
        if (live) {
#pragma unroll
            for (int q = 0; q < 16; ++q) acc[q] += (double)(v[q].x * v[q].x + v[q].y * v[q].y);
        }
    }
    // fftshift: bin k of the transform is entry (k + P/2) mod P of the estimate
#pragma unroll
    for (int q = 0; q < 16; ++q) atomicAdd(&p.psd[(size_t)blockIdx.y * P + ((t + q * TPF + P / 2) & (P - 1))], acc[q]);
}

template <int N> size_t psd_masked_smem() {
    using PP = FftPlan<8 * N>;
    return ((size_t)PP::NTW + (size_t)(256 / PP::TPF) * PP::XLEN) * sizeof(float2);
}

// one batch's frames of all n_spec spectra (their product already in Y) into psd: about two CTAs per SM in all
template <int N> cudaError_t psd_masked_launch(const DeviceCtx& d, PsdMaskedParams p, int n_spec) {
    const size_t sm = psd_masked_smem<N>();
    const cudaError_t e = cudaFuncSetAttribute(psd_masked_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return e;
    const int gx = (int)std::min<long long>(p.items, std::max(1, 2 * d.sm_count / n_spec));
    psd_masked_kernel<N><<<dim3(gx, n_spec), 256, sm, d.stream>>>(p);
    return cudaGetLastError();
}

// The Tx side of a wofdm_ber_run_masked job; the Rx fields are not read
int check_masked_tx(wofdm_ctx* h, const wofdm_sys_t* s, int roll_off) {
    if (!s) return fail(h, WOFDM_EINVAL, "sys is NULL");
    const int N = s->N;
    if (N != 128 && N != 256 && N != 512) return fail(h, WOFDM_EUNSUPPORTED, "the channel-mask variant is built for N = 128, 256, 512");
    if (s->bits != 2 && s->bits != 4 && s->bits != 6 && s->bits != 8) return fail(h, WOFDM_EINVAL, "bits must be 2, 4, 6 or 8 (square QAM)");
    if (s->S < 2) return fail(h, WOFDM_EINVAL, "S must be >= 2 (symbol 0 is the pilot)");
    if (s->cp < 0 || s->cp > N || s->cs < 0 || s->cs > N) return fail(h, WOFDM_EINVAL, "cp and cs must lie in [0, N]");
    const int n_tx = N + s->cp + s->cs, M = 2 * n_tx - 1;
    if (s->tail_tx < 0 || 2 * s->tail_tx > n_tx) return fail(h, WOFDM_EINVAL, "tail_tx must lie in [0, n_tx / 2]");
    if (s->constellation != 0 && s->constellation != 1) return fail(h, WOFDM_EINVAL, "constellation must be 0 or 1");
    if (s->precision != 0 && s->precision != 1) return fail(h, WOFDM_EINVAL, "precision must be 0 (fp32) or 1 (fp64)");
    if (s->guard < 0 || 2 * s->guard >= N) return fail(h, WOFDM_EINVAL, "guard must lie in [0, N/2)");
    if (s->guard > 0 && s->bits == 8) return fail(h, WOFDM_EUNSUPPORTED, "a guard band needs bits < 8 (constellation byte 255 marks a null sub-carrier)");
    if (s->precision != 0) return fail(h, WOFDM_EUNSUPPORTED, "the channel-mask variant runs in fp32");
    if (roll_off < 1 || M / 2 + 2 * roll_off > M) return fail(h, WOFDM_EINVAL, "roll_off does not fit the mask");
    if (2 * n_tx > 3 * N + 1) return fail(h, WOFDM_EUNSUPPORTED, "cp + cs too long for the mask kernel (n_tx <= 1.5 N)");
    return WOFDM_OK;
}

}  // namespace
}  // namespace wofdm

using namespace wofdm;

extern "C" int wofdm_psd_masked(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, int roll_off, uint64_t seed,
                                int64_t f0, int64_t n_frames, int estimator, double* psd_masked, double* psd_unmasked) {
    return wofdm_psd_masked_multi(h, sys, win_tx, &roll_off, 1, seed, f0, n_frames, estimator, psd_masked, psd_unmasked);
}

extern "C" int wofdm_psd_masked_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const int* roll_off,
                                      int n_var, uint64_t seed, int64_t f0, int64_t n_frames, int estimator, double* psd_masked,
                                      double* psd_unmasked) {
    NvtxRange nvtx_("wofdm_psd_masked");
    if (!h) return WOFDM_EINVAL;
    if (!win_tx) return fail(h, WOFDM_EINVAL, "win_tx is NULL");
    if (!psd_masked && !psd_unmasked) return fail(h, WOFDM_EINVAL, "both outputs are NULL");
    if (f0 < 0 || n_frames < 1 || f0 > INT64_MAX - n_frames) return fail(h, WOFDM_EINVAL, "bad frame range (f0 >= 0, n_frames >= 1, no overflow)");
    if (estimator != 0 && estimator != 1) return fail(h, WOFDM_EINVAL, "estimator must be 0 (reference) or 1 (Hann, 50 % overlap)");
    if (n_var < 1 || n_var > WOFDM_MAX_VARIANTS) return fail(h, WOFDM_EINVAL, "n_var must be in [1, WOFDM_MAX_VARIANTS]");
    if (!roll_off) return fail(h, WOFDM_EINVAL, "NULL roll_off");
    int rc = WOFDM_OK;
    for (int v = 0; v < n_var && !rc; ++v) rc = check_masked_tx(h, sys, roll_off[v]);
    if (rc) return rc;
    const int N = sys->N, P = 8 * N, n_tx = N + sys->cp + sys->cs, stride = n_tx - sys->tail_tx;
    const long long len = (long long)sys->tail_tx + (long long)sys->S * stride;
    if (len < P) return fail(h, WOFDM_EINVAL, "stream shorter than one periodogram slice (tail_tx + S * stride < 8N)");
    if (len > INT32_MAX / 2) return fail(h, WOFDM_EINVAL, "stream too long");
    const int hop = estimator == 1 ? P / 2 : P;
    const int n_slices = estimator == 1 ? (int)((len - P) / hop) + 1 : (int)(len / P) + 1;   // (the reference adds the remainder slice)
    const int G = 256 / (P / 16), groups = (n_slices + G - 1) / G;

    DeviceCtx& d = h->devs[0];
    WOFDM_CUDA(h, cudaSetDevice(d.dev));
    // batches of about `cols` symbols.  An L2-resident batch (16 384 symbols, 40 MB of Y at N = 256) measured slower than
    // 131 072 (DESIGN.md 4b): the product's tail wave and the launches per batch cost more than re-reading Y from HBM
    const long long cols = 131072;
    const long long batch = std::min<long long>(n_frames, std::max<long long>(1, cols / sys->S));
    // the spectra as pairs of one product: the masked ones (window v, roll_off[v]), then the unmasked ones (window v, a unit
    // impulse); spectrum k goes to outs[k]
    std::vector<float> wf;
    std::vector<int> ro;
    std::vector<double*> outs;
    for (int half = 0; half < 2; ++half) {
        double* o = half == 0 ? psd_masked : psd_unmasked;
        if (!o) continue;
        for (int v = 0; v < n_var; ++v) {
            const std::vector<double> wd = tx_table(*sys, win_tx + (size_t)v * n_tx, false);
            wf.insert(wf.end(), wd.begin(), wd.end());
            ro.push_back(half == 0 ? roll_off[v] : 0);
            outs.push_back(o + (size_t)v * P);
        }
    }
    const int n_spec = (int)outs.size();
    const std::vector<double> twd = build_twiddles(P);
    const std::vector<float> twf(twd.begin(), twd.end());
    MaskGemm mg;
    const size_t need = wf.size() * 4 + twf.size() * 4 + (size_t)n_spec * P * 8 + mask_gemm_plan(*sys, batch, n_spec, mg);
    rc = arena_reserve(h, d, need);
    if (rc) return rc;
    float* d_w = static_cast<float*>(arena_take(d, wf.size() * 4));
    float2* d_twp = static_cast<float2*>(arena_take(d, twf.size() * 4));
    double* d_psd = static_cast<double*>(arena_take(d, (size_t)n_spec * P * 8));
    if (!d_w || !d_twp || !d_psd) return fail(h, WOFDM_ENOMEM, "arena exhausted");
    WOFDM_CUDA(h, cudaMemcpyAsync(d_w, wf.data(), wf.size() * 4, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(d_twp, twf.data(), twf.size() * 4, cudaMemcpyHostToDevice, d.stream));
    WOFDM_CUDA(h, cudaMemsetAsync(d_psd, 0, (size_t)n_spec * P * 8, d.stream));

    auto run = [&]() -> int {
        const int r = mask_gemm_setup(h, d, mg, ro.data(), d_w);
        if (r) return r;
        PsdMaskedParams p;
        memset(&p, 0, sizeof(p));
        p.Y = mg.Y; p.ypair = mg.ypair; p.Yp = mg.Yp; p.S = sys->S; p.stride = stride; p.n_tx = n_tx; p.len = (int)len;
        p.n_slices = n_slices; p.groups = groups; p.hop = hop; p.hann = estimator == 1; p.twp = d_twp; p.psd = d_psd;
        for (long long fb = f0; fb < f0 + n_frames; fb += batch) {
            const long long nf = std::min(batch, f0 + n_frames - fb);
            const int rb = mask_gemm_batch(h, d, mg, seed, fb, nf);
            if (rb) return rb;
            p.items = nf * groups;
            cudaError_t e = cudaSuccess;
            switch (N) {
                case 128: e = psd_masked_launch<128>(d, p, n_spec); break;
                case 256: e = psd_masked_launch<256>(d, p, n_spec); break;
                default:  e = psd_masked_launch<512>(d, p, n_spec); break;
            }
            WOFDM_CUDA(h, e);
            h->launches += 1;
        }
        return WOFDM_OK;
    };
    rc = run();
    if (rc) {                                  // nothing of this call stays in flight
        cudaStreamSynchronize(d.stream);
        return rc;
    }
    std::vector<double> acc((size_t)n_spec * P);
    WOFDM_CUDA(h, cudaMemcpyAsync(acc.data(), d_psd, acc.size() * 8, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
    // mean periodogram; the Hann slices carry 8N / sum(w^2) = 8/3, so a white stream reads the same level under both estimators
    const double scale = (estimator == 1 ? 8.0 / 3.0 : 1.0) / ((double)n_slices * (double)n_frames);
    for (int k = 0; k < n_spec; ++k)
        for (int i = 0; i < P; ++i) outs[k][i] = acc[(size_t)k * P + i] * scale;
    return WOFDM_OK;
}
