// wofdm_capi.cu -- C-ABI: context management, parameter table, window builders.
#include <cstring>
#include <new>

#include "host_common.h"

namespace wofdm {

int arena_reserve(wofdm_ctx* h, DeviceCtx& d, size_t bytes) {
    bytes += 64 * 256;   // alignment slack for up to 64 sub-allocations
    if (bytes > d.arena_cap) {
        WOFDM_CUDA(h, cudaSetDevice(d.dev));
        if (d.arena) {
            WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
            WOFDM_CUDA(h, cudaFree(d.arena));
            d.arena = nullptr;
            d.arena_cap = 0;
        }
        size_t cap = bytes + bytes / 4;
        WOFDM_CUDA(h, cudaMalloc(&d.arena, cap));
        d.arena_cap = cap;
    }
    d.arena_used = 0;
    return WOFDM_OK;
}

void* arena_take(DeviceCtx& d, size_t bytes) {
    size_t off = (d.arena_used + 255) & ~(size_t)255;
    if (off + bytes > d.arena_cap) return nullptr;
    d.arena_used = off + bytes;
    return static_cast<char*>(d.arena) + off;
}

double qam_scale(const wofdm_sys_t& s) {
    if (s.constellation == 0) return 1.0;
    const double M = (double)(1 << s.bits);
    return 1.0 / std::sqrt(2.0 * (M - 1.0) / 3.0);
}

int validate_sys(wofdm_ctx* h, const wofdm_sys_t* s, int L) {
    if (!s) return fail(h, WOFDM_EINVAL, "sys is NULL");
    if (s->N < 16 || s->N > 1024 || (s->N & (s->N - 1))) return fail(h, WOFDM_EINVAL, "N must be a power of two in [16, 1024]");
    if (s->bits != 2 && s->bits != 4 && s->bits != 6 && s->bits != 8) return fail(h, WOFDM_EINVAL, "bits must be 2, 4, 6 or 8 (square QAM)");
    if (s->S < 2) return fail(h, WOFDM_EINVAL, "S must be >= 2 (symbol 0 is the pilot)");
    if (s->cp < 0 || s->cp > s->N || s->cs < 0 || s->cs > s->N) return fail(h, WOFDM_EINVAL, "cp and cs must lie in [0, N]");
    if (s->tail_tx < 0 || s->tail_rx < 0 || (s->tail_rx & 1)) return fail(h, WOFDM_EINVAL, "tails must be >= 0 and tail_rx even");
    if (s->rm < 0 || s->shift < 0 || s->shift >= s->N) return fail(h, WOFDM_EINVAL, "rm must be >= 0 and shift in [0, N)");
    const int n_tx = s->N + s->cp + s->cs, n_rx = s->N + s->tail_rx + s->rm;
    if (n_rx != n_tx - s->tail_tx) return fail(h, WOFDM_EINVAL, "inconsistent system: N+tail_rx+rm != N+cp+cs-tail_tx");
    if (2 * s->tail_tx > n_tx) return fail(h, WOFDM_EINVAL, "tail_tx too long for the Tx block");
    if (s->tail_rx > s->N) return fail(h, WOFDM_EINVAL, "tail_rx too long");
    if (s->noise_norm != 0 && s->noise_norm != 1) return fail(h, WOFDM_EINVAL, "noise_norm must be 0 or 1");
    if (s->constellation != 0 && s->constellation != 1) return fail(h, WOFDM_EINVAL, "constellation must be 0 or 1");
    if (s->precision != 0 && s->precision != 1) return fail(h, WOFDM_EINVAL, "precision must be 0 (fp32) or 1 (fp64)");
    if (s->guard < 0 || 2 * s->guard >= s->N) return fail(h, WOFDM_EINVAL, "guard must lie in [0, N/2)");
    if (s->guard > 0 && s->bits == 8) return fail(h, WOFDM_EUNSUPPORTED, "a guard band needs bits < 8 (constellation byte 255 marks a null sub-carrier)");
    if (L < 1 || L > 4096) return fail(h, WOFDM_EINVAL, "L must lie in [1, 4096]");
    return WOFDM_OK;
}

std::vector<double> build_twiddles(int N) {
    int a = 0, n = N;
    while (n % 16 == 0 && n >= 16) { n /= 16; ++a; }
    const int r = n;
    std::vector<double> tw;
    const double two_pi = 6.283185307179586476925286766559;
    int Ns = 16;
    for (int p = 1; p < a; ++p, Ns *= 16) {
        if (p == 1) {                        // rows of TW1_PITCH = 18: thread k's factors m = 0..15 side by side (fft_regs.cuh)
            for (int k = 0; k < 16; ++k)
                for (int m = 0; m < wofdm::TW1_PITCH; ++m) {
                    const double ang = m < 16 ? -two_pi * (double)(k * m) / 256.0 : 0.0;
                    tw.push_back(m < 16 ? std::cos(ang) : 0.0);
                    tw.push_back(m < 16 ? std::sin(ang) : 0.0);
                }
            continue;
        }
        for (int m = 0; m < 16; ++m)
            for (int k = 0; k < Ns; ++k) {
                const double ang = -two_pi * (double)(k * m) / (double)(16 * Ns);
                tw.push_back(std::cos(ang));
                tw.push_back(std::sin(ang));
            }
    }
    if (r > 1)
        for (int m = 0; m < r; ++m)
            for (int j = 0; j < N / r; ++j) {
                const double ang = -two_pi * (double)((long long)j * m) / (double)N;
                tw.push_back(std::cos(ang));
                tw.push_back(std::sin(ang));
            }
    return tw;
}

static void rc_tail(int t, std::vector<double>& out) {
    // sin^2(pi/2 * (1/2 + a/t)), a = -(t-1)/2 ... (t-1)/2   (transmitter.py:81-82, receiver.py:52-53)
    out.resize(t);
    for (int k = 0; k < t; ++k) {
        const double a = (double)k - (double)(t - 1) / 2.0;
        const double s = std::sin(3.14159265358979323846 / 2.0 * (0.5 + a / (double)t));
        out[k] = s * s;
    }
}

}  // namespace wofdm

using namespace wofdm;

extern "C" {

int wofdm_version(void) { return WOFDM_VERSION; }

int wofdm_device_count(int* n) {
    if (!n) return WOFDM_EINVAL;
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { *n = 0; cudaGetLastError(); return WOFDM_ENODEV; }
    *n = c;
    return WOFDM_OK;
}

int wofdm_create_on(wofdm_handle* out, const int* device_ids, int n) {
    if (!out || !device_ids || n < 1) return WOFDM_EINVAL;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { cudaGetLastError(); return WOFDM_ENODEV; }
    wofdm_ctx* h = new (std::nothrow) wofdm_ctx();
    if (!h) return WOFDM_ENOMEM;
    for (int i = 0; i < n; ++i) {
        if (device_ids[i] < 0 || device_ids[i] >= count) { delete h; return WOFDM_ENODEV; }
        DeviceCtx d;
        d.dev = device_ids[i];
        cudaDeviceProp prop;
        if (cudaSetDevice(d.dev) != cudaSuccess || cudaGetDeviceProperties(&prop, d.dev) != cudaSuccess ||
            cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError();
            delete h;
            return WOFDM_ECUDA;
        }
        if (prop.major < 10) { delete h; return WOFDM_ENODEV; }   // sm_100a code only
        d.sm_count = prop.multiProcessorCount;
        d.smem_optin = prop.sharedMemPerBlockOptin;
        h->devs.push_back(d);
    }
    register_ber_f32_tconv(h->variants);
    register_ber_f32_tconv2(h->variants);
    register_ber_f32_tconv2_hs(h->variants);
    register_ber_f32_regs(h->variants);
    register_ber_f32_staged(h->variants);
    register_ber_f64_staged(h->variants);
    register_ber_f32_tconv2_res(h->variants);
    register_ber_staged_res(h->variants);
    register_ber_f32_regs_res(h->variants);
    register_ber_f32_tconv2_txy_res(h->variants);
    register_ber_f32_regs_txs_res(h->variants);
    *out = h;
    return WOFDM_OK;
}

int wofdm_create(wofdm_handle* out, int n_gpus) {
    if (!out || n_gpus < 0) return WOFDM_EINVAL;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { cudaGetLastError(); *out = nullptr; return WOFDM_ENODEV; }
    if (n_gpus == 0) n_gpus = count;
    if (n_gpus > count) { *out = nullptr; return WOFDM_ENODEV; }
    std::vector<int> ids(n_gpus);
    for (int i = 0; i < n_gpus; ++i) ids[i] = i;
    return wofdm_create_on(out, ids.data(), n_gpus);
}

int wofdm_destroy(wofdm_handle h) {
    if (!h) return WOFDM_EINVAL;
    for (auto& d : h->devs) {
        cudaSetDevice(d.dev);
        if (d.stream) { cudaStreamSynchronize(d.stream); cudaStreamDestroy(d.stream); }
        if (d.arena) cudaFree(d.arena);
    }
    if (!h->devs.empty()) cudaSetDevice(h->devs[0].dev);
    for (auto& e : h->interf_ev)
        if (e) cudaEventDestroy(e);
    for (auto& e : h->hess_ev)
        if (e) cudaEventDestroy(e);
    delete h;
    return WOFDM_OK;
}

const char* wofdm_last_error(wofdm_handle h) { return h ? h->err.c_str() : "invalid handle"; }

int64_t wofdm_launch_count(wofdm_handle h) { return h ? h->launches : -1; }

int wofdm_params_from_name(const char* name, int N, int cp, int tail_tx, int tail_rx, wofdm_sys_t* out) {
    if (!name || !out) return WOFDM_EINVAL;
    const int hh = tail_rx / 2;
    int cs, rm, shift;
    if (!strcmp(name, "CP")) { cs = 0; rm = cp; shift = 0; }
    else if (!strcmp(name, "wtx")) { cs = tail_tx; rm = cp; shift = 0; }
    else if (!strcmp(name, "CPwtx")) { cs = 0; rm = cp - tail_tx; shift = tail_tx; }
    else if (!strcmp(name, "wrx")) { cs = hh; rm = cp - hh; shift = 0; }
    else if (!strcmp(name, "CPwrx")) { cs = 0; rm = cp - tail_rx; shift = hh; }
    else if (!strcmp(name, "WOLA")) { cs = tail_tx; rm = cp - tail_rx; shift = hh; }
    else if (!strcmp(name, "CPW")) { cs = tail_tx + hh; rm = cp - hh; shift = 0; }
    else return WOFDM_EINVAL;
    out->N = N; out->cp = cp; out->cs = cs; out->tail_tx = tail_tx; out->tail_rx = tail_rx;
    out->rm = rm; out->shift = shift;
    return WOFDM_OK;
}

int wofdm_rc_window_tx(const wofdm_sys_t* s, double* out) {
    if (!s || !out) return WOFDM_EINVAL;
    const int n_tx = s->N + s->cp + s->cs, b = s->tail_tx;
    if (2 * b > n_tx) return WOFDM_EINVAL;
    std::vector<double> t;
    rc_tail(b, t);
    for (int i = 0; i < n_tx; ++i) out[i] = 1.0;
    for (int i = 0; i < b; ++i) { out[i] = t[i]; out[n_tx - 1 - i] = t[i]; }
    return WOFDM_OK;
}

int wofdm_rc_window_rx(const wofdm_sys_t* s, double* out) {
    if (!s || !out) return WOFDM_EINVAL;
    const int n = s->N + s->tail_rx, d = s->tail_rx;
    if (d > s->N) return WOFDM_EINVAL;
    std::vector<double> t;
    rc_tail(d, t);
    for (int i = 0; i < n; ++i) out[i] = 1.0;
    for (int i = 0; i < d; ++i) { out[i] = t[i]; out[n - 1 - i] = t[i]; }
    return WOFDM_OK;
}

int wofdm_expand_window_tx(const wofdm_sys_t* s, const double* x, double* out) {
    // w = [x[b..1], x0 * ones(n_tx - 2b), x[1..b]]   (optimization_tools/utils.py:13-43)
    if (!s || !x || !out) return WOFDM_EINVAL;
    const int n_tx = s->N + s->cp + s->cs, b = s->tail_tx;
    if (2 * b > n_tx) return WOFDM_EINVAL;
    for (int i = 0; i < n_tx; ++i) out[i] = x[0];
    for (int i = 1; i <= b; ++i) { out[b - i] = x[i]; out[n_tx - b + i - 1] = x[i]; }
    return WOFDM_OK;
}

int wofdm_expand_window_rx(const wofdm_sys_t* s, const double* x, double* out) {
    // w = [x0 - x[1..h], x[h..1], x0 * ones(N - d), x[1..h], x0 - x[h..1]]   (utils.py:46-73)
    if (!s || !x || !out) return WOFDM_EINVAL;
    const int d = s->tail_rx, hh = d / 2, N = s->N;
    if ((d & 1) || d > N) return WOFDM_EINVAL;
    for (int i = 0; i < N + d; ++i) out[i] = x[0];
    for (int i = 1; i <= hh; ++i) {
        out[i - 1] = x[0] - x[i];
        out[2 * hh - i] = x[i];
        out[N + i - 1] = x[i];
        out[N + d - i] = x[0] - x[i];
    }
    return WOFDM_OK;
}

}  // extern "C"
