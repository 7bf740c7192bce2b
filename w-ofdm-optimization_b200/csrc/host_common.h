// host_common.h -- context, error plumbing and small host helpers behind the C-ABI.
#pragma once
#include <cuda_runtime.h>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/wofdm.h"
#include "ber_registry.h"

namespace wofdm {

struct DeviceCtx {
    int dev = 0;
    cudaStream_t stream = nullptr;
    int sm_count = 0;
    size_t smem_optin = 0;
    // grow-only staging arena for the host-pointer entry points (no cudaMalloc per call)
    void* arena = nullptr;
    size_t arena_cap = 0, arena_used = 0;
};

}  // namespace wofdm

struct wofdm_ctx {
    std::vector<wofdm::DeviceCtx> devs;
    std::vector<wofdm::BerVariant> variants;
    std::string err;
    int64_t launches = 0;
    // device time of the last wofdm_interf_power* call (CUDA events on the handle's stream): whole call on the device
    // (uploads, builders, band product, contraction, download), the band product and the contraction alone; -1 = not taken
    cudaEvent_t interf_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    double interf_ms[3] = {-1.0, -1.0, -1.0};
    double interf_k_isi = 0.0, interf_kp = 0.0;      // K rows contracted per ISI slice / per slice 0
    // last wofdm_window_hessian* call: device time (uploads to download, CUDA events), host time of the channel-set
    // factorisation, passes of the device pipeline (virtual channels); -1 / 0 = not taken
    cudaEvent_t hess_ev[2] = {nullptr, nullptr};
    double hess_ms = -1.0, hess_factor_ms = 0.0;
    int hess_passes = 0;
};

namespace wofdm {

// NVTX range around a C-ABI entry point (header-only NVTX v3: a no-op unless a profiler is attached)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

inline int fail(wofdm_ctx* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    return code;
}

#define WOFDM_CUDA(h, expr)                                                                         \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            return ::wofdm::fail((h), e__ == cudaErrorMemoryAllocation ? WOFDM_ENOMEM : WOFDM_ECUDA, \
                                 std::string(#expr) + ": " + cudaGetErrorString(e__));              \
        }                                                                                           \
    } while (0)

// bump allocation out of the device's arena; invalidated by arena_reset()
int arena_reserve(wofdm_ctx* h, DeviceCtx& d, size_t bytes);
void* arena_take(DeviceCtx& d, size_t bytes);
inline void arena_reset(DeviceCtx& d) { d.arena_used = 0; }

int validate_sys(wofdm_ctx* h, const wofdm_sys_t* s, int L);
double qam_scale(const wofdm_sys_t& s);
inline int noise_len(const wofdm_sys_t& s, int L) {
    const int stride = s.N + s.cp + s.cs - s.tail_tx;
    return s.noise_norm == 0 ? s.S * stride : s.tail_tx + s.S * stride + L - 1;
}

// FFT twiddle sections in the layout fft_regs.cuh documents, as interleaved doubles (re, im)
std::vector<double> build_twiddles(int N);

}  // namespace wofdm
