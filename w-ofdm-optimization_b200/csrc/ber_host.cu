// ber_host.cu -- host side of K1: variant selection, device tables, plans, and the
// wofdm_ber_* entry points of include/wofdm.h.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <new>

#include "host_common.h"
#include "mask_kernel.cuh"
#include "mask_gemm.h"
#include "ber_tconv2.cuh"

using namespace wofdm;

struct PlanDev {
    void *d_wtx = nullptr, *d_wrx = nullptr, *d_tw = nullptr, *d_chan = nullptr, *d_snr = nullptr;
    unsigned long long* d_cnt = nullptr;
    long long* d_seg = nullptr;    // segment table of wofdm_ber_run_segments / _adaptive (BerParams::seg): [seg_cap][4]
    void* d_scratch = nullptr;
    size_t scratch_bytes = 0;
    int blocks_per_sm = 0;
    long long max_ctas = 0;
    bool pending = false;
    cudaStream_t last_stream = nullptr;
};

struct wofdm_ber_plan_s {
    wofdm_ctx* ctx = nullptr;
    wofdm_sys_t sys{};
    int L = 0, C = 0, n_snr = 0;
    const BerVariant* var = nullptr;
    BerSmem lay{};
    int chunk = 0, use_global = 0;
    int flat_tx = 0, flat_rx = 0;  // bit v = window pair v
    int n_var = 1;                 // window pairs of the plan
    bool fused = false;            // all of them in ONE launch (second-generation tensor-core kernel); else one launch each
    bool transient = false;    // buffers live in the devices' arenas (one-shot plan of wofdm_ber_run*): nothing to free
    // resolved counters (wofdm_ber_run_resolved): WOFDM_BY_* flags, 0 for the plans of the public plan API.  The kernel that
    // production picks for the same arguments fixes the noise numbering (chunk, split, n48): noise_var; else noise_var == var
    int resolve = 0;
    const BerVariant* noise_var = nullptr;
    size_t cnt_per_var = 0;        // u64 counters of one window pair: [cells][bins][2] (unresolved: [n_snr][2])
    int seg_cap = 0;               // entries of the devices' segment tables (PlanDev::d_seg), 0: none
    std::vector<PlanDev> devs;
};

std::vector<double> wofdm::tx_table(const wofdm_sys_t& s, const double* win_tx, bool unit_peak) {
    const int n_tx = s.N + s.cp + s.cs;
    double k = qam_scale(s) / (double)s.N;   // IDFT 1/N (transmitter.py:58) and constellation scale
    if (unit_peak) {
        double mx = 0.0;
        for (int i = 0; i < n_tx; ++i) mx = std::max(mx, std::fabs(win_tx[i]));
        if (mx > 0.0 && std::isfinite(mx)) k /= mx;
    }
    std::vector<double> a(n_tx);
    for (int i = 0; i < n_tx; ++i) a[i] = win_tx[i] * k;
    return a;
}

namespace {

struct Choice {
    const BerVariant* var = nullptr;
    BerSmem lay{};
    int chunk = 0, use_global = 0;
};

// a Tx window that is one non-zero value between its tails, which lie inside the prefix and the suffix
bool flat_tx_window(const wofdm_sys_t& s, const double* wt) {
    const int n_tx = s.N + s.cp + s.cs;
    bool ft = s.cp >= s.tail_tx && s.cs >= s.tail_tx && wt[s.tail_tx] != 0.0;
    for (int i = s.tail_tx; ft && i < n_tx - s.tail_tx; ++i) ft = wt[i] == wt[s.tail_tx];
    return ft;
}

// where a kernel takes the Tx stream from: drawn in the kernel, read from HBM (BerParams::tx_stream, BerVariant::txs), or
// gathered from the mask product's output (BerParams::tx_y, BerVariant::txy)
enum class TxSource { drawn, stream, gather };

// WOFDM_VARIANT: `want` occurs in `name`; with a trailing '$', at its end
bool variant_name_matches(const char* name, const char* want) {
    const size_t nw = strlen(want);
    if (nw == 0 || want[nw - 1] != '$') return strstr(name, want) != nullptr;
    const size_t nn = strlen(name);
    return nw - 1 <= nn && strncmp(name + nn - (nw - 1), want, nw - 1) == 0;
}

// what a caller of choose_variant asks for
struct KernelRequest {
    bool verify = false;              // the verify instantiations (wofdm_ber_verify)
    bool staged_only = false;
    bool no_tconv = false;            // no tensor-core kernels
    bool no_circ = false;             // no circular-interior kernels
    const double* win_tx = nullptr;   // Tx window whose flatness the circular-interior and HS kernels need; NULL: neither
    int nvar = 1;                     // window pairs per launch
    TxSource tx = TxSource::drawn;
};

// the shape class of the fixed-shape tensor-core kernels (ber_tconv2.cuh: HS): one window pair with a flat Tx window
// (BerParams::flat_tx), no Rx window tails, no guard band, symbols drawn in the kernel (no Tx stream from the mask chain)
bool tconv2_fixed_shape(const wofdm_sys_t& s, const KernelRequest& rq) {
    return rq.win_tx != nullptr && rq.nvar == 1 && rq.tx == TxSource::drawn && s.tail_rx == 0 && s.guard == 0 &&
           flat_tx_window(s, rq.win_tx);
}

// ... and the geometry compiled into a fixed-shape instance (ber_tconv2.cuh: tconv2_geom(geom)), L the job's channel length
bool tconv2_fixed_geometry(const wofdm_sys_t& s, int L, int geom) {
    const Tconv2Geom g = tconv2_geom(geom);
    return g.N > 0 && s.N == g.N && s.S == g.S && s.cp == g.cp && s.cs == g.cs && s.tail_tx == g.tail_tx && s.tail_rx == 0 &&
           s.rm == g.rm && s.shift == g.shift && L == g.L && s.bits == g.bits;
}

// tensor-core kernel: windows that are one value between their tails (BerParams::flat_tx / flat_rx)
// (n_var window pairs back to back: bit v of flat_tx / flat_rx = pair v)
void fill_flat(BerParams& prm, const wofdm_sys_t& s, const double* win_tx, const double* win_rx, int n_var = 1) {
    const int n_tx = s.N + s.cp + s.cs, n_wr = s.N + s.tail_rx;
    prm.flat_tx = prm.flat_rx = 0;
    for (int v = 0; v < n_var; ++v) {
        const double* wt = win_tx + (size_t)v * n_tx;
        const double* wr = win_rx + (size_t)v * n_wr;
        const bool ft = flat_tx_window(s, wt);
        bool fr = wr[s.tail_rx] != 0.0;
        for (int i = s.tail_rx; fr && i < s.N; ++i) fr = wr[i] == wr[s.tail_rx];
        prm.flat_tx |= (ft ? 1 : 0) << v;
        prm.flat_rx |= (fr ? 1 : 0) << v;
    }
}

// noise numbering of a frame shared by a cluster (BerParams::split)
void fill_split(BerParams& prm, const BerVariant& v) {
    prm.split = v.CL > 1 ? prm.S * prm.stride / v.CL : 0;
    prm.split_nt = v.CL > 1 ? v.NT : 0;
    prm.n48 = v.ntile > 0 ? 1 : 0;     // 48-bit noise draws in receiver layout (ber_kernel.cuh: noise_draw48)
}

// the staged kernel (verify / resolved-counter instance) of the frame's N and precision, with noise block `chunk`: frame
// buffers in shared memory where they fit, else in global memory (use_global)
int choose_staged(wofdm_ctx* h, const wofdm_sys_t& s, int L, size_t smem_cap, bool verify, bool res, int chunk, Choice* out) {
    const int stride = s.N + s.cp + s.cs - s.tail_tx;
    for (const auto& v : h->variants) {
        if (v.TC != 0 || v.fp64 != (s.precision == 1) || v.verify != verify || v.res != res || v.N != s.N) continue;
        Choice c;
        c.var = &v;
        c.chunk = chunk;
        c.lay = v.layout(s.S, stride, s.tail_tx, s.tail_rx, L, 0, 0);
        if (c.lay.bytes > smem_cap) {
            c.use_global = 1;
            c.lay = v.layout(s.S, stride, s.tail_tx, s.tail_rx, L, 0, 1);
            if (c.lay.bytes > smem_cap) return fail(h, WOFDM_EUNSUPPORTED, "frame does not fit the staged kernel's shared memory");
        }
        *out = c;
        return WOFDM_OK;
    }
    return fail(h, WOFDM_EUNSUPPORTED, res ? "no compiled resolved-counter kernel for this N / precision"
                                           : "no compiled kernel variant for this N / precision");
}

// The kernel of request rq, among those without resolved counters (BerVariant::res): a tensor-core kernel wherever one
// applies, else a register kernel, else the staged kernel.  WOFDM_NO_TCONV and WOFDM_NO_CIRC add no_tconv / no_circ;
// WOFDM_VARIANT=<substring> restricts the tensor-core and register candidates (kernel tuning aid, e.g. "_b2"); a trailing
// '$' anchors it at the end of the name ("tiles9_b2$": the generic kernel, not its fixed-shape instances).
int choose_variant(wofdm_ctx* h, const wofdm_sys_t& s, int L, size_t smem_cap, const KernelRequest& rq, Choice* out) {
    const int stride = s.N + s.cp + s.cs - s.tail_tx;
    const int sec = s.S * stride;
    const bool want_txs = rq.tx != TxSource::drawn, want_txy = rq.tx == TxSource::gather;
    const bool no_tconv = rq.no_tconv || getenv("WOFDM_NO_TCONV");
    const char* want = getenv("WOFDM_VARIANT");
    bool flat = rq.win_tx != nullptr && !rq.no_circ && !getenv("WOFDM_NO_CIRC");
    if (flat)
        for (int i = s.tail_tx; i < s.N + s.cp + s.cs - s.tail_tx; ++i)
            if (rq.win_tx[i] != rq.win_tx[s.tail_tx]) { flat = false; break; }
    const bool fixed_shape = tconv2_fixed_shape(s, rq);
    Choice best;
    if (s.precision != 1 && !rq.staged_only) {
        for (const auto& v : h->variants) {
            if (v.TC == 0 || v.fp64 || v.verify != rq.verify || v.N != s.N || v.res) continue;
            if (want && !variant_name_matches(v.name, want)) continue;
            if (v.ntile > 0) {
                // channel convolution on the tensor cores (ber_tconv2.cuh): first choice wherever it applies -- one Tx pass,
                // L <= LB, prefix / suffix / tails inside the outer register rows, power sums and the zeros behind the
                // stream inside the frame's tiles.  Takes tx_stream too.
                // CL CTAs share a frame: S/CL consecutive symbols each, in one Tx pass of the CTA
                if (s.S % v.CL != 0) continue;
                const int tpf = s.N / 16, S_cta = s.S / v.CL, sec_cta = sec / v.CL, body = s.tail_tx + sec_cta;
                if (no_tconv || S_cta > v.NT / tpf || L > v.LB) continue;
                if (v.txy != want_txy) continue;                     // (the mask product's consumers serve the channel-mask variant only)
                if (v.fixed_shape && !fixed_shape) continue;
                if (v.geom > 0 && !tconv2_fixed_geometry(s, L, v.geom)) continue;
                if (v.CL > 1 && want_txs) continue;                  // (the masked Tx stream is a one-CTA-per-frame feature)
                // a receiver thread holds at most N48_MAXLEV noise samples besides its 16 FFT rows
                if ((stride - s.N + (s.noise_norm == 1 ? s.tail_tx + L - 1 : 0) + tpf - 1) / tpf > (v.LB > TCV_LB ? N48_MAXLEV : N48_MAXLEV_SHORT)) continue;
                if (s.cp > 2 * tpf || s.cs > 2 * tpf || s.tail_tx > 2 * tpf || s.tail_rx / 2 > tpf || s.shift > tpf) continue;
                const int need = std::max(s.noise_norm == 1 ? body + L - 1 : sec_cta, body + tconv2_zero(v.LB));
                if (need > 512 * v.ntile || sec_cta <= 512 * (v.ntile - 2)) continue;   // (the kernel range-checks its last two tiles only)
                const BerSmem lay = v.layout(S_cta, stride, s.tail_tx, s.tail_rx, L, rq.nvar, 0);
                if (lay.bytes > smem_cap) continue;
                // fewest taps of history first (MMAs per tile), then fewest tiles, then the fixed-geometry instance, then the
                // fixed-shape one (same noise numbering and arithmetic, counters bit for bit: DESIGN.md section 3)
                auto fixed_rank = [](const BerVariant& x) { return x.geom > 0 ? 2 : x.fixed_shape ? 1 : 0; };
                if (!best.var || best.var->ntile == 0 || v.LB < best.var->LB ||
                    (v.LB == best.var->LB && (v.ntile < best.var->ntile ||
                                              (v.ntile == best.var->ntile && fixed_rank(v) > fixed_rank(*best.var))))) {
                    best.var = &v; best.lay = lay; best.chunk = 0;
                }
                continue;
            }
            if (best.var && best.var->ntile > 0) continue;
            if (v.txs != want_txs) continue;                 // the tx_stream instantiations serve the channel-mask variant only
            // CL CTAs share a frame: S/CL consecutive symbols each, all of them in one pass of the CTA
            if (s.S % v.CL != 0 || (v.CL > 1 && s.S / v.CL > v.NT / (v.N / 16))) continue;
            const int S_cta = s.S / v.CL, sec_cta = sec / v.CL;
            const int chunk = ((sec_cta + v.NT - 1) / v.NT) | 1;
            if (chunk > v.TC || L > v.LB) continue;
            // the tuned kernels only look at the outer register rows for the prefix / suffix / heads / overlap-add
            // (ber_kernel.cuh, ER): rows are N/16 samples wide
            const int tpf = s.N / 16;
            if (s.cp > 2 * tpf || s.cs > 2 * tpf || s.tail_tx > 2 * tpf || s.tail_rx / 2 > tpf || s.shift > tpf) continue;
            if (v.full && !(chunk == v.TC && v.NT * v.TC == sec_cta)) continue;
            // circular interior: flat window, the tail_tx + L - 1 edge outputs of a symbol two per thread, one Tx pass
            if (v.circ && !(flat && s.tail_tx + L - 1 <= 2 * tpf && s.S <= v.NT / tpf && s.cp + 2 * tpf >= s.tail_tx + L - 1)) continue;
            const BerSmem lay = v.layout(S_cta, stride, s.tail_tx, s.tail_rx, L, chunk, 0);
            if (lay.bytes > smem_cap) continue;
            // measured order (DESIGN.md section 3): the exact-fit direct kernel, then the circular-interior kernels
            // (+8 % over a direct kernel whose chunk does not fit exactly, -2..+1 % against the exact fit), then the rest
            auto rank = [](const BerVariant& x) { return (x.full && !x.circ) ? 0 : x.circ ? 1 : 2; };
            const bool better = !best.var || rank(v) < rank(*best.var) ||
                                (rank(v) == rank(*best.var) && (v.TC < best.var->TC || (v.TC == best.var->TC && v.full && !best.var->full)));
            if (better) { best.var = &v; best.lay = lay; best.chunk = chunk; }
        }
    }
    if (!best.var) return choose_staged(h, s, L, smem_cap, rq.verify, false, ((sec + 255) / 256) | 1, out);   // (noise block B of the staged policy: any odd number)
    *out = best;
    return WOFDM_OK;
}

// Resolved counters: the twin of the kernel `prod` that wofdm_ber_run_multi (or the channel-mask chain) picks -- the
// resolved-counter instance with the same key (BerVariant::key: same arithmetic, same noise blocks) -- where its
// accumulators fit (fused: all n_var pairs in one launch, else one launch per pair); else the staged twin, which numbers
// its noise like `prod` through noise_at (BerParams::chunk / split / n48).  *fused_out: the twin evaluates all pairs in one
// launch.
int choose_resolved(wofdm_ctx* h, const wofdm_sys_t& s, int L, size_t smem_cap, const Choice& prod, bool fused, int n_var,
                    Choice* out, bool* fused_out) {
    const BerVariant& p = *prod.var;
    const int stride = s.N + s.cp + s.cs - s.tail_tx;
    *fused_out = false;
    const bool staged_only = getenv("WOFDM_RESOLVED_STAGED") != nullptr;   // test aid: the staged twin with production's numbering
    if (p.TC > 0 && !staged_only) {
        for (const auto& v : h->variants) {
            if (!v.res || v.verify || v.key() != p.key()) continue;
            // tensor-core twins: all pairs in one launch where the accumulators of all of them fit, else one launch per pair
            // (same counters); register twins: production's noise block
            for (int nv : {fused ? n_var : 1, 1}) {
                const BerSmem lay = v.layout(s.S / v.CL, stride, s.tail_tx, s.tail_rx, L, v.ntile > 0 ? nv : prod.chunk, 0);
                if (lay.bytes > smem_cap) continue;
                out->var = &v; out->lay = lay; out->chunk = prod.chunk; out->use_global = 0;
                *fused_out = fused && nv == n_var;
                return WOFDM_OK;
            }
            break;
        }
    }
    return choose_staged(h, s, L, smem_cap, false, true, prod.chunk, out);
}

template <typename T> void cast_vec(const std::vector<double>& src, std::vector<unsigned char>& dst) {
    dst.resize(src.size() * sizeof(T));
    T* p = reinterpret_cast<T*>(dst.data());
    for (size_t i = 0; i < src.size(); ++i) p[i] = (T)src[i];
}
void cast_any(bool fp64, const std::vector<double>& src, std::vector<unsigned char>& dst) {
    if (fp64) cast_vec<double>(src, dst); else cast_vec<float>(src, dst);
}

// the device inputs of a job in the kernels' precision, shared by plans, the verify path and the channel-mask chain
struct HostTables {
    std::vector<unsigned char> wtx, wrx, tw, chan, snr;
    size_t bytes() const { return wtx.size() + wrx.size() + tw.size() + chan.size() + snr.size(); }
};

// channel matrix L x C column-major complex double -> [C][L] V2<T> (same memory order, cast only).  unit_peak (tensor-core
// kernels, see build_tables): every channel's taps are divided by their largest component magnitude.
void cast_chan(bool fp64, const double* chan, size_t n_complex, std::vector<unsigned char>& dst, int L, bool unit_peak) {
    std::vector<double> v(chan, chan + 2 * n_complex);
    if (unit_peak) {
        for (size_t c = 0; c + (size_t)L <= n_complex; c += (size_t)L) {
            double mx = 0.0;
            for (int i = 0; i < 2 * L; ++i) mx = std::max(mx, std::fabs(v[2 * c + i]));
            if (mx > 0.0 && std::isfinite(mx)) {
                const double inv = 1.0 / mx;
                for (int i = 0; i < 2 * L; ++i) v[2 * c + i] *= inv;
            }
        }
    }
    cast_any(fp64, v, dst);
}

// The tables of n_var window pairs (back to back), the twiddles, C channels of L taps and n_snr SNR points (linear).
// unit_peak (tensor-core kernels): every Tx window is divided by its largest magnitude.  Those kernels stage the stream and
// the taps as fp16 pairs behind fixed power-of-two scales (ber_tconv.cuh: TCV_XSCALE, TCV_HSCALE), so their inputs must
// have a known range; the chain itself does not care -- a common factor of the Tx signal or of a channel's taps scales
// r, the noise follows the measured signal power (wofdm_simulation.py:135-138) and the pilot equaliser divides it out (:223-232).
HostTables build_tables(const wofdm_sys_t& s, const double* win_tx, const double* win_rx, int n_var, const double* chan, int L,
                        int C, const double* snr_db, int n_snr, bool unit_peak) {
    const bool fp64 = s.precision == 1;
    const int n_tx = s.N + s.cp + s.cs, n_wr = s.N + s.tail_rx;
    std::vector<double> a((size_t)n_var * n_tx), b(win_rx, win_rx + (size_t)n_var * n_wr);
    for (int v = 0; v < n_var; ++v) {
        const std::vector<double> wt = tx_table(s, win_tx + (size_t)v * n_tx, unit_peak);
        std::copy(wt.begin(), wt.end(), a.begin() + (size_t)v * n_tx);
    }
    std::vector<double> lin(n_snr);
    for (int i = 0; i < n_snr; ++i) lin[i] = std::pow(10.0, -0.1 * snr_db[i]);   // wofdm_simulation.py:138
    HostTables t;
    cast_any(fp64, a, t.wtx);
    cast_any(fp64, b, t.wrx);
    cast_any(fp64, build_twiddles(s.N), t.tw);
    cast_chan(fp64, chan, (size_t)L * C, t.chan, L, unit_peak);
    cast_any(fp64, lin, t.snr);
    return t;
}

// an arena block of max(bytes, 16) on device d, filled from src (unless NULL) on d's stream
cudaError_t arena_put(DeviceCtx& d, const void* src, size_t bytes, void** dst) {
    *dst = arena_take(d, std::max<size_t>(bytes, 16));
    if (!*dst) return cudaErrorMemoryAllocation;
    return src ? cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, d.stream) : cudaSuccess;
}

void fill_sys(BerParams& p, const wofdm_sys_t& s, int L) {
    memset(&p, 0, sizeof(p));
    p.N = s.N; p.cp = s.cp; p.cs = s.cs; p.tail_tx = s.tail_tx; p.tail_rx = s.tail_rx; p.rm = s.rm;
    p.shift = s.shift; p.bits = s.bits; p.S = s.S;
    p.n_tx = s.N + s.cp + s.cs;
    p.stride = p.n_tx - s.tail_tx;
    p.L = L;
    p.noise_norm = s.noise_norm; p.constellation = s.constellation;
    p.guard = s.guard;
    p.noise_len = noise_len(s, L);
    p.qscale = qam_scale(s);
}

// max_ctas: CTAs of this variant that can be resident on the device at once (a multiple of the cluster size)
int prepare_kernel(wofdm_ctx* h, const BerVariant& v, size_t smem, int sm_count, int* blocks_per_sm, long long* max_ctas) {
    WOFDM_CUDA(h, cudaFuncSetAttribute(v.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int nb = 0;
    WOFDM_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, v.fn, v.launch_threads, smem));
    if (v.ntile > 0) {
        // the occupancy calculator counts a kernel that allocates tensor memory as one CTA per SM; these kernels take
        // 256 of the 512 columns (N = 256; all of them at N = 512), so registers, shared memory and tensor memory together decide
        cudaFuncAttributes fa;
        int dev = 0, smem_sm = 0, regs_sm = 0;
        WOFDM_CUDA(h, cudaFuncGetAttributes(&fa, v.fn));
        WOFDM_CUDA(h, cudaGetDevice(&dev));
        WOFDM_CUDA(h, cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
        WOFDM_CUDA(h, cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev));
        const int by_smem = (int)((size_t)smem_sm / (smem + 1024)), by_regs = regs_sm / (((fa.numRegs + 7) & ~7) * v.launch_threads);
        const int by_tmem = 512 / (int)tconv_tmem_cols(v.ntile);
        nb = std::max(nb, std::min(by_smem, std::min(by_regs, by_tmem)));
    }
    if (getenv("WOFDM_DEBUG")) fprintf(stderr, "[wofdm] %s: smem %zu B, %d CTAs/SM\n", v.name, smem, nb);
    if (nb < 1) return fail(h, WOFDM_EUNSUPPORTED, "kernel variant cannot be resident on this device");
    *blocks_per_sm = nb;
    long long cap = (long long)nb * sm_count;
    if (v.CL > 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(v.CL * sm_count); cfg.blockDim = dim3(v.launch_threads); cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = v.CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int ncl = 0;
        WOFDM_CUDA(h, cudaOccupancyMaxActiveClusters(&ncl, v.fn, &cfg));
        if (ncl < 1) return fail(h, WOFDM_EUNSUPPORTED, "no thread-block cluster of this variant fits the device");
        // (tensor-memory kernels: the cluster occupancy query, too, counts one CTA per SM; nb above is the real residency.
        //  A grid larger than what is resident is still correct -- frames are taken round-robin by cluster index.)
        cap = std::max<long long>((long long)ncl * v.CL, v.ntile > 0 ? ((long long)nb * sm_count / v.CL) * v.CL : 0);
    }
    if (max_ctas) *max_ctas = cap;
    return WOFDM_OK;
}

size_t elem_bytes(const wofdm_sys_t& s) { return s.precision == 1 ? sizeof(double2) : sizeof(float2); }

// ---- argument checks of the wofdm_ber_* entry points ---------------------------------------------------------------------
// (each call keeps its own order of them: validate_sys and the channel-mask checks can return WOFDM_EUNSUPPORTED, the
//  others WOFDM_EINVAL, so the order decides the code of a call with several faults)

int check_shard(wofdm_ctx* h, int shard_index, int shard_count) {
    if (shard_count < 1 || shard_index < 0 || shard_index >= shard_count) return fail(h, WOFDM_EINVAL, "bad shard");
    return WOFDM_OK;
}

// resolve: WOFDM_BY_* flags; nonzero: at least one of them
int check_resolve(wofdm_ctx* h, int resolve, bool nonzero) {
    if ((nonzero && resolve == 0) || (resolve & ~(WOFDM_BY_SUBCARRIER | WOFDM_BY_CHANNEL)))
        return fail(h, WOFDM_EINVAL, nonzero ? "resolve must be a non-empty combination of WOFDM_BY_SUBCARRIER and WOFDM_BY_CHANNEL"
                                             : "resolve must be a combination of WOFDM_BY_SUBCARRIER and WOFDM_BY_CHANNEL");
    return WOFDM_OK;
}

int check_shape(wofdm_ctx* h, const wofdm_sys_t* sys, int L, int C, int n_snr, int n_var) {
    const int rc = validate_sys(h, sys, L);
    if (rc) return rc;
    if (C < 1 || n_snr < 1) return fail(h, WOFDM_EINVAL, "C and n_snr must be >= 1");
    if (n_var < 1 || n_var > WOFDM_MAX_VARIANTS) return fail(h, WOFDM_EINVAL, "n_var must be in [1, WOFDM_MAX_VARIANTS]");
    return WOFDM_OK;
}

// the frame ids of a job, n_snr * C * ensemble of them, must be representable
int check_frames(wofdm_ctx* h, int n_snr, int C, int64_t ensemble) {
    int64_t frames = 0;
    if (__builtin_mul_overflow((int64_t)n_snr, (int64_t)C, &frames) || __builtin_mul_overflow(frames, ensemble, &frames))
        return fail(h, WOFDM_EINVAL, "n_snr * C * ensemble overflows int64");
    return WOFDM_OK;
}

// a job of the main chain (ensemble: ensemble_max of the segment calls) and this process's shard of it
int check_job(wofdm_ctx* h, const wofdm_sys_t* sys, int L, int C, int n_snr, int n_var, int64_t ensemble, int shard_index,
              int shard_count) {
    int rc = check_shard(h, shard_index, shard_count);
    if (rc) return rc;
    if (ensemble < 1) return fail(h, WOFDM_EINVAL, "ensemble must be >= 1");
    rc = check_shape(h, sys, L, C, n_snr, n_var);
    return rc ? rc : check_frames(h, n_snr, C, ensemble);
}

// counters [n_var][n_snr][Cr][Nr] of `resolve`, 16 bytes each on the device: all of it must be representable
int check_counters(wofdm_ctx* h, const wofdm_sys_t& s, int C, int n_snr, int n_var, int resolve) {
    const int Cr = (resolve & WOFDM_BY_CHANNEL) ? C : 1, Nr = (resolve & WOFDM_BY_SUBCARRIER) ? s.N : 1;
    size_t n = 0, bytes = 0;
    if (__builtin_mul_overflow((size_t)n_snr, (size_t)Cr, &n) || __builtin_mul_overflow(n, (size_t)Nr, &n) ||
        __builtin_mul_overflow(n, (size_t)n_var, &n) || __builtin_mul_overflow(n, (size_t)16, &bytes) || n > (size_t)INT64_MAX / 16)
        return fail(h, WOFDM_EINVAL, "resolved counter array too large");
    return WOFDM_OK;
}

// a job of the channel-mask chain (one window pair, fp32, N = 128, 256 or 512, a mask that fits) and this process's shard
// of it; outputs_ok: the caller's output pointers are all non-NULL
int check_masked(wofdm_ctx* h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, const double* chan, int L,
                 int C, const double* snr_db, int n_snr, int64_t ensemble, int roll_off, int shard_index, int shard_count,
                 int resolve, bool outputs_ok) {
    int rc = check_shape(h, sys, L, C, n_snr, 1);
    if (rc) return rc;
    if (!win_tx || !win_rx || !chan || !snr_db || !outputs_ok) return fail(h, WOFDM_EINVAL, "NULL buffer");
    if (ensemble < 1) return fail(h, WOFDM_EINVAL, "ensemble must be >= 1");
    if (sys->precision != 0) return fail(h, WOFDM_EUNSUPPORTED, "the channel-mask variant runs in fp32");
    const int N = sys->N, n_tx = N + sys->cp + sys->cs, M = 2 * n_tx - 1;
    if (N != 128 && N != 256 && N != 512) return fail(h, WOFDM_EUNSUPPORTED, "the channel-mask variant is built for N = 128, 256, 512");
    if (roll_off < 1 || M / 2 + 2 * roll_off > M) return fail(h, WOFDM_EINVAL, "roll_off does not fit the mask");
    if (2 * n_tx > 3 * N + 1) return fail(h, WOFDM_EUNSUPPORTED, "cp + cs too long for the mask kernel (n_tx <= 1.5 N)");
    rc = check_shard(h, shard_index, shard_count);
    if (!rc) rc = check_frames(h, n_snr, C, ensemble);
    return rc ? rc : check_counters(h, *sys, C, n_snr, 1, resolve);
}

// check_masked for n_var window pairs with roll-offs roll_off[n_var] (the pairs differ only in what check_masked reads of
// roll_off), and their counters [n_var][n_snr][Cr][Nr]
int check_masked_multi(wofdm_ctx* h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, const double* chan,
                       int L, int C, const double* snr_db, int n_snr, int64_t ensemble, const int* roll_off, int n_var,
                       int shard_index, int shard_count, int resolve, bool outputs_ok) {
    if (n_var < 1 || n_var > WOFDM_MAX_VARIANTS) return fail(h, WOFDM_EINVAL, "n_var must be in [1, WOFDM_MAX_VARIANTS]");
    if (!roll_off) return fail(h, WOFDM_EINVAL, "NULL roll_off");
    for (int v = 0; v < n_var; ++v) {
        const int rc = check_masked(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble, roll_off[v], shard_index,
                                    shard_count, resolve, outputs_ok);
        if (rc) return rc;
    }
    return check_counters(h, *sys, C, n_snr, n_var, resolve);
}

// segments[n_seg][3] of a job: inside [0, n_snr) x [0, ensemble_max), e_count >= 1, no two segments of one point overlap
int check_segments(wofdm_ctx* h, const int64_t* segments, int n_seg, int n_snr, int64_t ensemble_max) {
    if (!segments || n_seg < 1) return fail(h, WOFDM_EINVAL, "segments must be a non-empty list");
    std::vector<std::pair<int64_t, int64_t>> iv((size_t)n_seg);
    for (int k = 0; k < n_seg; ++k) {
        const int64_t si = segments[3 * k], e0 = segments[3 * k + 1], ec = segments[3 * k + 2];
        if (si < 0 || si >= n_snr || e0 < 0 || e0 >= ensemble_max || ec < 1 || ec > ensemble_max - e0)
            return fail(h, WOFDM_EINVAL, "segment outside [0, n_snr) x [0, ensemble_max) or with e_count < 1");
        iv[k] = {si * ensemble_max + e0, ec};       // (< n_snr * ensemble_max: no overflow, checked by the caller)
    }
    std::sort(iv.begin(), iv.end());
    for (int k = 1; k < n_seg; ++k)
        if (iv[k].first < iv[k - 1].first + iv[k - 1].second) return fail(h, WOFDM_EINVAL, "overlapping segments of one SNR point");
    return WOFDM_OK;
}

// the stopping rule's own arguments (wofdm_ber_run_adaptive / wofdm_ber_run_masked_adaptive)
int check_target(wofdm_ctx* h, int target_kind, int64_t target, int64_t first_block, int shard_count, wofdm_reduce_fn reduce) {
    if (target_kind != WOFDM_TARGET_BIT_ERRORS && target_kind != WOFDM_TARGET_SYMBOL_ERRORS) return fail(h, WOFDM_EINVAL, "unknown target_kind");
    if (target < 1) return fail(h, WOFDM_EINVAL, "target must be >= 1");
    if (first_block < 1) return fail(h, WOFDM_EINVAL, "first_block must be >= 1");
    if (shard_count > 1 && !reduce) return fail(h, WOFDM_EINVAL, "shard_count > 1 needs a reduce callback (the schedule needs the job's counts)");
    return WOFDM_OK;
}

// ---- frame sets, shards and totals -----------------------------------------------------------------------------------------

// A list of segments {snr_idx, e_begin, e_count} (every channel of point snr_idx at ensemble indices [e_begin, e_begin +
// e_count)) as the devices read it (BerParams::seg): tab[k] = {g0, snr_idx, e_begin, e_count}, g0 the local index of
// segment k's first frame (segments in order, channel-major, then e); n_local frames in all.
struct Segments {
    std::vector<long long> tab;
    long long n_local = 0;
    int n() const { return (int)(tab.size() / 4); }
};

Segments seg_table(const int64_t* seg, int n_seg, int C) {
    Segments s;
    s.tab.resize((size_t)n_seg * 4);
    for (int k = 0; k < n_seg; ++k) {
        long long* t = &s.tab[4 * (size_t)k];
        t[0] = s.n_local; t[1] = seg[3 * k]; t[2] = seg[3 * k + 1]; t[3] = seg[3 * k + 2];
        s.n_local += (long long)C * seg[3 * k + 2];
    }
    return s;
}

// the segments {(si, 0, counts[si]) : si < n_snr}.  With counts[si] = ensemble: the whole job of a fixed call, whose local
// index is exactly the global frame id (si*C + c)*ensemble + e.
Segments job_segments(int C, const std::vector<int64_t>& counts) {
    std::vector<int64_t> seg;
    for (size_t si = 0; si < counts.size(); ++si) { seg.push_back((int64_t)si); seg.push_back(0); seg.push_back(counts[si]); }
    return seg_table(seg.data(), (int)counts.size(), C);
}

// The local indices of a frame set that one shard (shard_index, shard_count) owns: strided, j = shard_index (mod
// shard_count), the main chain's rule; or contiguous, the block [floor(n k / W), floor(n (k+1) / W)) of the n local
// indices, the channel-mask chain's rule.
struct ShardRule {
    bool contiguous;
    long long index, count;                // strided
    long long lo, hi;                      // contiguous: [lo, hi)
    static ShardRule strided(int index, int count) { return {false, index, count, 0, 0}; }
    static ShardRule block(long long n, int index, int count) {
        return {true, index, count, (long long)((__int128)n * index / count), (long long)((__int128)n * (index + 1) / count)};
    }
    // this shard's local indices in [a, b)
    long long frames(long long a, long long b) const {
        if (contiguous) return std::max(0LL, std::min(hi, b) - std::max(lo, a));
        auto upto = [&](long long x) -> long long { return x > index ? (x - index + count - 1) / count : 0; };
        return upto(b) - upto(a);
    }
};

// this shard's frames per counter cell (si, c) [n_snr][Cr] of a segment list: Cr = C (by channel) or 1
std::vector<long long> cell_frames(const Segments& sg, int n_snr, int C, int Cr, const ShardRule& r) {
    std::vector<long long> frames((size_t)n_snr * Cr, 0);
    for (int k = 0; k < sg.n(); ++k) {
        const long long g0 = sg.tab[4 * k], si = sg.tab[4 * k + 1], ec = sg.tab[4 * k + 3];
        const long long w = Cr > 1 ? ec : C * ec;      // local indices of one cell: one channel's, or all of them
        for (int c = 0; c < Cr; ++c) frames[(size_t)si * Cr + c] += r.frames(g0 + c * w, g0 + (c + 1) * w);
    }
    return frames;
}

// totals of counter cells [n_snr][Cr][Nr] from the frames of each cell (si, c): S-1 symbols per active bin and frame, 0 on
// guard bins; Nr == 1: every active bin of the frame.  bit_tot (may be NULL) = sym_tot * bits.
void cell_totals(const wofdm_sys_t& s, const std::vector<long long>& frames, int Nr, int64_t* sym_tot, int64_t* bit_tot) {
    const long long active = s.N - 2 * s.guard;
    for (size_t cell = 0; cell < frames.size(); ++cell) {
        int64_t* out = sym_tot + cell * Nr;
        if (Nr == 1) { out[0] = frames[cell] * active * (s.S - 1); continue; }
        for (int k = 0; k < Nr; ++k) {
            const int cc = (k + Nr / 2) & (Nr - 1);                   // ber_kernel.cuh: bin_active
            out[k] = (cc >= s.guard && cc < Nr - s.guard) ? frames[cell] * (s.S - 1) : 0;
        }
    }
    if (bit_tot)
        for (size_t i = 0; i < frames.size() * Nr; ++i) bit_tot[i] = sym_tot[i] * s.bits;
}

}  // namespace

// transient = true: device buffers come out of the per-device arena (no cudaMalloc / cudaFree per call); such a plan
// must be destroyed before the arena is used again (wofdm_ber_run_shard does exactly that)
// resolve != 0 (WOFDM_BY_* flags): counters [n_var][n_snr * Cr][Nr][2] in a buffer of their own (wofdm_ber_run_resolved)
// seg_cap > 0 (frame segments): the resolved twin runs even with resolve == 0 (counters [n_var][n_snr][2]) and every
// device gets a segment table of seg_cap entries (BerParams::seg)
static int plan_create_impl(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                            const double* chan, int L, int C, const double* snr_db, int n_snr,
                            wofdm_ber_plan* out, bool transient, int resolve = 0, int seg_cap = 0) {
    NvtxRange nvtx_("wofdm_ber_plan_create");
    if (!h) return WOFDM_EINVAL;
    if (!out) return fail(h, WOFDM_EINVAL, "plan out pointer is NULL");
    *out = nullptr;
    int rc = check_shape(h, sys, L, C, n_snr, n_var);
    if (rc) return rc;
    if (!win_tx || !win_rx || !chan || !snr_db) return fail(h, WOFDM_EINVAL, "NULL input buffer");

    wofdm_ber_plan_s* p = new (std::nothrow) wofdm_ber_plan_s();
    if (!p) return fail(h, WOFDM_ENOMEM, "host allocation failed");
    p->ctx = h; p->sys = *sys; p->L = L; p->C = C; p->n_snr = n_snr; p->transient = transient; p->n_var = n_var;
    p->seg_cap = seg_cap;
    Choice ch;
    size_t cap = h->devs[0].smem_optin;
    for (auto& d : h->devs) cap = std::min(cap, d.smem_optin);
    // several window pairs: one launch for all of them where the second-generation tensor-core kernel applies and holds
    // their tables; otherwise the pairs are launched one after the other on the same draws (same counters either way)
    {
        KernelRequest rq;
        rq.win_tx = win_tx;
        rq.nvar = n_var;
        rc = choose_variant(h, *sys, L, cap, rq, &ch);
    }
    p->fused = rc == WOFDM_OK && n_var > 1 && ch.var->ntile > 0;
    // (one launch per pair: no Tx window is passed, so no kernel that relies on the flatness of pair 0's is chosen)
    if (n_var > 1 && !p->fused) {
        KernelRequest rq;
        rq.no_circ = true;
        rc = choose_variant(h, *sys, L, cap, rq, &ch);
    }
    if (rc) { delete p; return rc; }
    p->noise_var = ch.var;
    p->cnt_per_var = (size_t)n_snr * 2;
    if (resolve || seg_cap > 0) {
        Choice rch;
        bool rfused = false;
        rc = choose_resolved(h, *sys, L, cap, ch, p->fused, n_var, &rch, &rfused);
        if (rc) { delete p; return rc; }
        ch.var = rch.var; ch.lay = rch.lay; ch.use_global = rch.use_global;     // (ch.chunk: the noise block of production)
        p->fused = rfused;
        p->resolve = resolve;
        p->cnt_per_var = (size_t)n_snr * ((resolve & WOFDM_BY_CHANNEL) ? C : 1) * ((resolve & WOFDM_BY_SUBCARRIER) ? sys->N : 1) * 2;
    }
    p->var = ch.var; p->lay = ch.lay; p->chunk = ch.chunk; p->use_global = ch.use_global;
    {
        BerParams fp;
        fill_flat(fp, *sys, win_tx, win_rx, n_var);
        p->flat_tx = fp.flat_tx; p->flat_rx = fp.flat_rx;
    }

    const HostTables t = build_tables(*sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, p->var->ntile > 0);

    p->devs.resize(h->devs.size());
    for (size_t i = 0; i < h->devs.size(); ++i) {
        DeviceCtx& d = h->devs[i];
        PlanDev& pd = p->devs[i];
        auto dev_alloc = [&](void** dst, size_t bytes) -> cudaError_t {
            if (!transient) return cudaMalloc(dst, std::max<size_t>(bytes, 16));
            *dst = arena_take(d, std::max<size_t>(bytes, 16));
            return *dst ? cudaSuccess : cudaErrorMemoryAllocation;
        };
        auto up = [&](void** dst, const std::vector<unsigned char>& src) -> cudaError_t {
            cudaError_t e = dev_alloc(dst, src.size());
            if (e != cudaSuccess) return e;
            return cudaMemcpyAsync(*dst, src.data(), src.size(), cudaMemcpyHostToDevice, d.stream);
        };
        cudaError_t e = cudaSetDevice(d.dev);
        if (e == cudaSuccess) {
            rc = prepare_kernel(h, *p->var, p->lay.bytes, d.sm_count, &pd.blocks_per_sm, &pd.max_ctas);
            if (rc) { const std::string msg = h->err; wofdm_ber_plan_destroy(p); h->err = msg; return rc; }
        }
        // staged policy with frame buffers in global memory: two of them per resident CTA
        const size_t scratch_elems = (size_t)p->lay.pad + sys->tail_tx + (size_t)sys->S * (sys->N + sys->cp + sys->cs - sys->tail_tx) + 64;
        pd.scratch_bytes = p->use_global ? (size_t)pd.blocks_per_sm * d.sm_count * 2 * scratch_elems * elem_bytes(*sys) : 0;
        if (e == cudaSuccess && transient) {
            rc = arena_reserve(h, d, t.bytes() + (resolve ? 0 : (size_t)n_var * n_snr * 16) + pd.scratch_bytes + (size_t)seg_cap * 32);
            if (rc) { const std::string msg = h->err; wofdm_ber_plan_destroy(p); h->err = msg; return rc; }
        }
        if (e == cudaSuccess) e = up(&pd.d_wtx, t.wtx);
        if (e == cudaSuccess) e = up(&pd.d_wrx, t.wrx);
        if (e == cudaSuccess) e = up(&pd.d_tw, t.tw);
        if (e == cudaSuccess) e = up(&pd.d_chan, t.chan);
        if (e == cudaSuccess) e = up(&pd.d_snr, t.snr);
        // (resolved counters: a buffer of their own, outside the arena -- it can be large, and failing to get it is WOFDM_ENOMEM)
        if (e == cudaSuccess && resolve) e = cudaMalloc(reinterpret_cast<void**>(&pd.d_cnt), n_var * p->cnt_per_var * sizeof(unsigned long long));
        else if (e == cudaSuccess) e = dev_alloc(reinterpret_cast<void**>(&pd.d_cnt), (size_t)n_var * n_snr * 2 * sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);   // host vectors go out of scope
        if (e == cudaSuccess && p->use_global) e = dev_alloc(&pd.d_scratch, pd.scratch_bytes);
        if (e == cudaSuccess && seg_cap > 0) e = dev_alloc(reinterpret_cast<void**>(&pd.d_seg), (size_t)seg_cap * 32);
        if (e != cudaSuccess) {
            std::string msg = std::string("plan upload: ") + cudaGetErrorString(e);
            wofdm_ber_plan_destroy(p);
            return fail(h, e == cudaErrorMemoryAllocation ? WOFDM_ENOMEM : WOFDM_ECUDA, msg);
        }
    }
    *out = p;
    return WOFDM_OK;
}

extern "C" {

int wofdm_ber_plan_create(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                          const double* chan, int L, int C, const double* snr_db, int n_snr,
                          wofdm_ber_plan* out) {
    return plan_create_impl(h, sys, win_tx, win_rx, 1, chan, L, C, snr_db, n_snr, out, false);
}

int wofdm_ber_plan_create_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                                const double* chan, int L, int C, const double* snr_db, int n_snr, wofdm_ber_plan* out) {
    return plan_create_impl(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, out, false);
}

int wofdm_ber_plan_variants(wofdm_ber_plan p, int* fused) {
    if (!p) return WOFDM_EINVAL;
    if (fused) *fused = p->fused ? 1 : 0;
    return p->n_var;
}

}  // extern "C"

// d_seg != nullptr (a twin plan): the launch runs the n_local frames of the segment table d_seg[n_seg][4] (BerParams::seg)
// instead of the n_snr * C * ensemble frames of the plan; ensemble is then the job's ensemble_max
static int plan_launch_impl(wofdm_ber_plan p, int slot, int64_t ensemble, uint64_t seed, uint32_t variant,
                            int shard_index, int shard_count, void* stream, void** d_counters,
                            const long long* d_seg = nullptr, int n_seg = 0, long long n_local = 0) {
    if (!p) return WOFDM_EINVAL;
    wofdm_ctx* h = p->ctx;
    if (slot < 0 || slot >= (int)p->devs.size()) return fail(h, WOFDM_EINVAL, "device slot out of range");
    if (ensemble < 1) return fail(h, WOFDM_EINVAL, "ensemble must be >= 1");
    if (shard_count < 1 || shard_index < 0 || shard_index >= shard_count) return fail(h, WOFDM_EINVAL, "bad shard");
    if (variant > 0xfffffff0u - WOFDM_MAX_VARIANTS) return fail(h, WOFDM_EINVAL, "variant too large");
    DeviceCtx& d = h->devs[slot];
    PlanDev& pd = p->devs[slot];
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d.stream;
    WOFDM_CUDA(h, cudaSetDevice(d.dev));

    const long long total = d_seg ? n_local : (long long)p->n_snr * p->C * ensemble;
    const long long mine = total > shard_index ? (total - shard_index + shard_count - 1) / shard_count : 0;
    BerParams prm;
    fill_sys(prm, p->sys, p->L);
    prm.chunk = p->chunk; prm.use_global = p->use_global;
    prm.flat_tx = p->flat_tx; prm.flat_rx = p->flat_rx;
    fill_split(prm, *p->noise_var);
    prm.res_chan = (p->resolve & WOFDM_BY_CHANNEL) ? 1 : 0;
    prm.res_bins = (p->resolve & WOFDM_BY_SUBCARRIER) ? 1 : 0;
    prm.seg = d_seg; prm.n_seg = n_seg;
    prm.win_tx = pd.d_wtx; prm.win_rx = pd.d_wrx; prm.tw = pd.d_tw; prm.chan = pd.d_chan; prm.snr_lin = pd.d_snr;
    prm.C = p->C; prm.n_snr = p->n_snr; prm.ensemble = ensemble;
    prm.seed = seed; prm.variant = variant;
    philox_round_keys(seed, prm.rk);
    prm.frame_begin = shard_index; prm.frame_step = shard_count; prm.n_frames = mine;
    prm.counters = pd.d_cnt;
    prm.scratch = pd.d_scratch;
    prm.scratch_elems = p->use_global ? (long long)(pd.scratch_bytes / ((size_t)pd.blocks_per_sm * d.sm_count * 2 * elem_bytes(p->sys))) : 0;

    // a launch owns its slot's counters: one that is still pending on ANOTHER stream must finish before they are zeroed
    if (pd.pending && pd.last_stream != st) WOFDM_CUDA(h, cudaStreamSynchronize(pd.last_stream));
    WOFDM_CUDA(h, cudaMemsetAsync(pd.d_cnt, 0, (size_t)p->n_var * p->cnt_per_var * sizeof(unsigned long long), st));
    if (mine > 0) {
        long long cap = pd.max_ctas;
        if (const char* lim = getenv("WOFDM_MAX_CTAS_PER_SM"))            // tuning aid: occupancy sensitivity
            cap = std::min<long long>(cap, (long long)std::max(1, atoi(lim)) * d.sm_count);
        const int cl = p->var->CL;
        const int grid = (int)std::min<long long>(mine, std::max<long long>(cap / cl, 1)) * cl;   // CTAs = frames in flight x cluster size
        if (p->fused || p->n_var == 1) {
            prm.nvar = p->n_var;
            WOFDM_CUDA(h, p->var->launch(prm, grid, p->lay.bytes, st));
            h->launches += 1;
        } else {
            // one launch per window pair: pair v = a single-pair launch with variant + v on tables / counters v
            const size_t eb = p->sys.precision == 1 ? sizeof(double) : sizeof(float);
            const int n_tx = p->sys.N + p->sys.cp + p->sys.cs, n_wr = p->sys.N + p->sys.tail_rx;
            for (int v = 0; v < p->n_var; ++v) {
                BerParams pv = prm;
                pv.nvar = 1;
                pv.win_tx = static_cast<const char*>(pd.d_wtx) + (size_t)v * n_tx * eb;
                pv.win_rx = static_cast<const char*>(pd.d_wrx) + (size_t)v * n_wr * eb;
                pv.flat_tx = (p->flat_tx >> v) & 1; pv.flat_rx = (p->flat_rx >> v) & 1;
                pv.variant = variant + (uint32_t)v;
                pv.counters = pd.d_cnt + (size_t)v * p->cnt_per_var;
                WOFDM_CUDA(h, p->var->launch(pv, grid, p->lay.bytes, st));
                h->launches += 1;
            }
        }
    }
    pd.pending = true;
    pd.last_stream = st;
    if (d_counters) *d_counters = pd.d_cnt;
    return WOFDM_OK;
}

// sum of the counter arrays of every slot launched since the last read -> bit_err / sym_err [n_var * cnt_per_var / 2]
// (the layout of the plan's counters with the {bit, sym} pair split)
static int read_counters(wofdm_ber_plan p, int64_t* bit_err, int64_t* sym_err) {
    wofdm_ctx* h = p->ctx;
    const size_t n_out = (size_t)p->n_var * p->cnt_per_var / 2;
    std::vector<unsigned long long> tmp;
    try { tmp.resize(n_out * 2); } catch (const std::bad_alloc&) { return fail(h, WOFDM_ENOMEM, "host allocation failed"); }
    for (size_t i = 0; i < n_out; ++i) { bit_err[i] = 0; sym_err[i] = 0; }
    for (size_t i = 0; i < p->devs.size(); ++i) {
        PlanDev& pd = p->devs[i];
        if (!pd.pending) continue;
        cudaError_t e = cudaSetDevice(h->devs[i].dev);
        if (e == cudaSuccess) e = cudaMemcpyAsync(tmp.data(), pd.d_cnt, n_out * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, pd.last_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(pd.last_stream);
        if (e != cudaSuccess) return fail(h, WOFDM_ECUDA, std::string("counters: ") + cudaGetErrorString(e));
        for (size_t k = 0; k < n_out; ++k) { bit_err[k] += (int64_t)tmp[2 * k]; sym_err[k] += (int64_t)tmp[2 * k + 1]; }
        pd.pending = false;
    }
    return WOFDM_OK;
}

extern "C" {

int wofdm_ber_plan_launch(wofdm_ber_plan p, int slot, int64_t ensemble, uint64_t seed, uint32_t variant,
                          int shard_index, int shard_count, void* stream, void** d_counters) {
    NvtxRange nvtx_("wofdm_ber_plan_launch");
    return plan_launch_impl(p, slot, ensemble, seed, variant, shard_index, shard_count, stream, d_counters);
}

int wofdm_ber_plan_read(wofdm_ber_plan p, int64_t* bit_err, int64_t* sym_err) {
    if (!p) return WOFDM_EINVAL;
    if (!bit_err || !sym_err) return fail(p->ctx, WOFDM_EINVAL, "NULL output buffer");
    return read_counters(p, bit_err, sym_err);        // [n_var][n_snr]
}

const char* wofdm_ber_plan_kernel(wofdm_ber_plan p) { return (p && p->var) ? p->var->name : ""; }

int wofdm_ber_plan_destroy(wofdm_ber_plan p) {
    if (!p) return WOFDM_EINVAL;
    for (size_t s = 0; s < p->devs.size(); ++s) {
        PlanDev& pd = p->devs[s];
        cudaSetDevice(p->ctx->devs[s].dev);
        if (pd.pending && pd.last_stream) cudaStreamSynchronize(pd.last_stream);
        if (p->resolve) cudaFree(pd.d_cnt);     // (its own buffer, also in a transient plan)
        if (p->transient) continue;             // arena memory
        cudaFree(pd.d_wtx); cudaFree(pd.d_wrx); cudaFree(pd.d_tw); cudaFree(pd.d_chan); cudaFree(pd.d_snr);
        if (!p->resolve) cudaFree(pd.d_cnt);
        cudaFree(pd.d_scratch);
        cudaFree(pd.d_seg);
    }
    cudaGetLastError();
    delete p;
    return WOFDM_OK;
}

}  // extern "C"

namespace {

// The schedule of include/wofdm.h for one point after a round that ran *block more ensemble indices of it: m = its fewest
// cumulative errors over the rows.  Returns true when the point is done; else *block is its next block.
bool schedule_step(int64_t m, int64_t target, int64_t ensemble_max, int64_t* used, int64_t* block) {
    *used += *block;
    if (m >= target || *used == ensemble_max) return true;
    // min(ensemble_max - e, 2b, m > 0 ? max(1, ceil((target - m) * e / m)) : 2b), exact in 128 bits, saturating
    __int128 nb = std::min<__int128>((__int128)ensemble_max - *used, (__int128)2 * *block);
    if (m > 0) {
        const __int128 need = ((__int128)(target - m) * *used + m - 1) / m;
        nb = std::min(nb, std::max<__int128>(1, need));
    }
    *block = (int64_t)nb;
    return false;
}

// One launch of plan p on every device of the handle, then the summed counters.  Device i takes the sub-shard
// shard_index + shard_count*i of shard_count*ndev, so results do not depend on the GPU count.  segs (twin plans): the
// launches run the local indices of that segment list, of a job of `ensemble` = ensemble_max indices, instead of the
// plan's whole job.
int run_plan(wofdm_ber_plan p, int64_t ensemble, uint64_t seed, uint32_t variant, int shard_index, int shard_count,
             const Segments* segs, int64_t* bit_err, int64_t* sym_err) {
    wofdm_ctx* h = p->ctx;
    const int nd = (int)h->devs.size();
    if (segs && segs->n() > p->seg_cap) return fail(h, WOFDM_EINVAL, "more segments than the plan's segment table holds");
    for (int i = 0; i < nd; ++i) {
        DeviceCtx& d = h->devs[i];
        PlanDev& pd = p->devs[i];
        if (segs) {
            WOFDM_CUDA(h, cudaSetDevice(d.dev));
            // (pageable source: the copy returns once the table is staged; the previous launch on this stream is ordered before it)
            WOFDM_CUDA(h, cudaMemcpyAsync(pd.d_seg, segs->tab.data(), segs->tab.size() * sizeof(long long), cudaMemcpyHostToDevice, d.stream));
        }
        const int rc = plan_launch_impl(p, i, ensemble, seed, variant, shard_index + shard_count * i, shard_count * nd, nullptr,
                                        nullptr, segs ? pd.d_seg : nullptr, segs ? segs->n() : 0, segs ? segs->n_local : 0);
        if (rc) return rc;
    }
    return read_counters(p, bit_err, sym_err);
}

// A checked job of the main chain on a one-shot plan: the whole job (segs == nullptr: the production kernels, or their
// resolved twins with resolve != 0) or the frames of a segment list (the twins).  -> counters [n_var][n_snr][Cr][Nr] and
// this shard's totals [n_snr][Cr][Nr]; bit_tot may be NULL.
int run_job(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var, const double* chan,
            int L, int C, const double* snr_db, int n_snr, int64_t ensemble, const Segments* segs, uint64_t seed, uint32_t variant,
            int shard_index, int shard_count, int resolve, int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot, int64_t* bit_tot) {
    wofdm_ber_plan p = nullptr;
    int rc = plan_create_impl(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, &p, true, resolve, segs ? segs->n() : 0);
    if (rc) return rc;
    rc = run_plan(p, ensemble, seed, variant, shard_index, shard_count, segs, bit_err, sym_err);
    wofdm_ber_plan_destroy(p);
    if (rc) return rc;
    const int Cr = (resolve & WOFDM_BY_CHANNEL) ? C : 1, Nr = (resolve & WOFDM_BY_SUBCARRIER) ? sys->N : 1;
    const Segments all = segs ? Segments() : job_segments(C, std::vector<int64_t>(n_snr, ensemble));
    cell_totals(*sys, cell_frames(segs ? *segs : all, n_snr, C, Cr, ShardRule::strided(shard_index, shard_count)), Nr, sym_tot, bit_tot);
    return WOFDM_OK;
}

// wofdm_ber_run_multi (resolve 0, bit_tot) and wofdm_ber_run_resolved (a checked resolve)
int run_fixed(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var, const double* chan,
              int L, int C, const double* snr_db, int n_snr, int64_t ensemble, uint64_t seed, uint32_t variant, int shard_index,
              int shard_count, int resolve, int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot, int64_t* bit_tot) {
    if (!bit_err || !sym_err || !sym_tot || (!resolve && !bit_tot)) return fail(h, WOFDM_EINVAL, "NULL output buffer");
    int rc = check_job(h, sys, L, C, n_snr, n_var, ensemble, shard_index, shard_count);
    if (!rc) rc = check_counters(h, *sys, C, n_snr, n_var, resolve);
    if (rc) return rc;
    return run_job(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, ensemble, nullptr, seed, variant, shard_index,
                   shard_count, resolve, bit_err, sym_err, sym_tot, bit_tot);
}

// The stopping rule of include/wofdm.h over `rows` rows of counters (wofdm_ber_run_adaptive / _masked_adaptive).  Each round
// runs the next block of every active point, in ascending SNR order, as one segment list: run_round gives this process's
// counters [rows][n_snr]; reduce (optional) sums them, packed [rows][n_snr][2] = {bit, sym}, over the processes; a point
// stops when its fewest errors over the rows reach the target.  Fills the call's outputs.
int run_adaptive(wofdm_ctx* h, const wofdm_sys_t& s, int C, int n_snr, int rows, int64_t ensemble_max, int64_t first_block,
                 int target_kind, int64_t target, wofdm_reduce_fn reduce, void* reduce_user,
                 const std::function<int(const Segments&, int64_t*, int64_t*)>& run_round, int64_t* ensemble_used,
                 int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot, int* rounds) {
    const size_t nr = (size_t)rows, ns = (size_t)n_snr;
    std::vector<int64_t> used(ns, 0), block(ns, std::min(first_block, ensemble_max)), rbit(nr * ns), rsym(nr * ns), red(nr * ns * 2);
    std::vector<int64_t> tbit(nr * ns, 0), tsym(nr * ns, 0);
    std::vector<char> done(ns, 0);
    int nround = 0;
    for (;;) {
        std::vector<int64_t> seg;
        for (size_t s = 0; s < ns; ++s)
            if (!done[s]) { seg.push_back((int64_t)s); seg.push_back(used[s]); seg.push_back(block[s]); }
        if (seg.empty()) break;
        const int rc = run_round(seg_table(seg.data(), (int)(seg.size() / 3), C), rbit.data(), rsym.data());
        if (rc) return rc;
        ++nround;
        for (size_t k = 0; k < nr * ns; ++k) { red[2 * k] = rbit[k]; red[2 * k + 1] = rsym[k]; }
        if (reduce && reduce(red.data(), (int64_t)red.size(), reduce_user) != 0) return fail(h, WOFDM_EINVAL, "the reduce callback failed");
        for (size_t k = 0; k < nr * ns; ++k) { tbit[k] += red[2 * k]; tsym[k] += red[2 * k + 1]; }
        const std::vector<int64_t>& t = target_kind == WOFDM_TARGET_BIT_ERRORS ? tbit : tsym;
        for (size_t s = 0; s < ns; ++s) {
            if (done[s]) continue;
            int64_t m = INT64_MAX;
            for (size_t r = 0; r < nr; ++r) m = std::min(m, t[r * ns + s]);
            done[s] = schedule_step(m, target, ensemble_max, &used[s], &block[s]);
        }
    }
    *rounds = nround;
    std::copy(used.begin(), used.end(), ensemble_used);
    std::copy(tbit.begin(), tbit.end(), bit_err);
    std::copy(tsym.begin(), tsym.end(), sym_err);
    // (the job's totals: every process ran the same schedule)
    cell_totals(s, cell_frames(job_segments(C, used), n_snr, C, 1, ShardRule::strided(0, 1)), 1, sym_tot, bit_tot);
    return WOFDM_OK;
}

}  // namespace

extern "C" {

int wofdm_ber_run_shard(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                        const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                        uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                        int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot) {
    return wofdm_ber_run_multi(h, sys, win_tx, win_rx, 1, chan, L, C, snr_db, n_snr, ensemble, seed, variant, shard_index,
                               shard_count, bit_err, bit_tot, sym_err, sym_tot);
}

int wofdm_ber_run_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                        const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                        uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                        int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_multi");
    if (!h) return WOFDM_EINVAL;
    return run_fixed(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, ensemble, seed, variant, shard_index, shard_count,
                     0, bit_err, sym_err, sym_tot, bit_tot);
}

int wofdm_ber_run_resolved(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                           const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                           uint64_t seed, uint32_t variant, int shard_index, int shard_count, int resolve,
                           int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_resolved");
    if (!h) return WOFDM_EINVAL;
    const int rc = check_resolve(h, resolve, true);
    if (rc) return rc;
    return run_fixed(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, ensemble, seed, variant, shard_index, shard_count,
                     resolve, bit_err, sym_err, sym_tot, nullptr);
}

int wofdm_ber_run_segments(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                           const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                           const int64_t* segments, int n_seg, uint64_t seed, uint32_t variant, int shard_index,
                           int shard_count, int resolve, int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_segments");
    if (!h) return WOFDM_EINVAL;
    int rc = check_resolve(h, resolve, false);
    if (rc) return rc;
    if (!bit_err || !sym_err || !sym_tot) return fail(h, WOFDM_EINVAL, "NULL output buffer");
    rc = check_job(h, sys, L, C, n_snr, n_var, ensemble_max, shard_index, shard_count);
    if (!rc) rc = check_segments(h, segments, n_seg, n_snr, ensemble_max);
    if (!rc) rc = check_counters(h, *sys, C, n_snr, n_var, resolve);
    if (rc) return rc;
    const Segments sg = seg_table(segments, n_seg, C);
    return run_job(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, ensemble_max, &sg, seed, variant, shard_index,
                   shard_count, resolve, bit_err, sym_err, sym_tot, nullptr);
}

int wofdm_ber_run_adaptive(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                           const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                           int64_t first_block, int target_kind, int64_t target, uint64_t seed, uint32_t variant,
                           int shard_index, int shard_count, wofdm_reduce_fn reduce, void* reduce_user,
                           int64_t* ensemble_used, int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot,
                           int* rounds) {
    NvtxRange nvtx_("wofdm_ber_run_adaptive");
    if (!h) return WOFDM_EINVAL;
    if (!ensemble_used || !bit_err || !bit_tot || !sym_err || !sym_tot || !rounds) return fail(h, WOFDM_EINVAL, "NULL output buffer");
    int rc = check_job(h, sys, L, C, n_snr, n_var, ensemble_max, shard_index, shard_count);
    if (!rc) rc = check_target(h, target_kind, target, first_block, shard_count, reduce);
    if (rc) return rc;
    wofdm_ber_plan p = nullptr;
    rc = plan_create_impl(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, &p, true, 0, n_snr);
    if (rc) return rc;
    rc = run_adaptive(h, *sys, C, n_snr, n_var, ensemble_max, first_block, target_kind, target, reduce, reduce_user,
                      [&](const Segments& sg, int64_t* be, int64_t* se) {
                          return run_plan(p, ensemble_max, seed, variant, shard_index, shard_count, &sg, be, se);
                      },
                      ensemble_used, bit_err, bit_tot, sym_err, sym_tot, rounds);
    wofdm_ber_plan_destroy(p);
    return rc;
}

int wofdm_ber_run(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                  const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                  uint64_t seed, uint32_t variant,
                  int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot) {
    return wofdm_ber_run_shard(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble, seed, variant, 0, 1,
                               bit_err, bit_tot, sym_err, sym_tot);
}

int wofdm_ber_verify(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                     const double* chan, int L, int F, const double* snr_db,
                     const int32_t* sym_idx, const double* noise, int variant_kernel,
                     double* eq_out, int32_t* dec_idx, int64_t* bit_err, int64_t* sym_err) {
    NvtxRange nvtx_("wofdm_ber_verify");
    if (!h) return WOFDM_EINVAL;
    int rc = validate_sys(h, sys, L);
    if (rc) return rc;
    if (!win_tx || !win_rx || !chan || !snr_db || !sym_idx || !noise || !eq_out || !dec_idx || !bit_err || !sym_err)
        return fail(h, WOFDM_EINVAL, "NULL buffer");
    if (F < 1) return fail(h, WOFDM_EINVAL, "F must be >= 1");
    const int M = 1 << sys->bits;
    const size_t n_sym = (size_t)sys->N * sys->S * F;
    for (size_t i = 0; i < n_sym; ++i)
        if (sym_idx[i] < 0 || sym_idx[i] >= M) return fail(h, WOFDM_EINVAL, "sym_idx entry outside the constellation");

    DeviceCtx& d = h->devs[0];
    WOFDM_CUDA(h, cudaSetDevice(d.dev));
    Choice ch;
    KernelRequest rq;
    rq.verify = true;
    rq.staged_only = variant_kernel == 1;
    rq.no_tconv = variant_kernel == 2 || variant_kernel == 3;
    rq.no_circ = variant_kernel == 2;
    rq.win_tx = win_tx;
    rc = choose_variant(h, *sys, L, d.smem_optin, rq, &ch);
    if (rc) return rc;
    int nb = 0;
    long long max_ctas = 0;
    rc = prepare_kernel(h, *ch.var, ch.lay.bytes, d.sm_count, &nb, &max_ctas);
    if (rc) return rc;
    const int grid = (int)std::min<long long>(F, std::max<long long>(max_ctas / ch.var->CL, 1)) * ch.var->CL;

    const HostTables t = build_tables(*sys, win_tx, win_rx, 1, chan, L, F, snr_db, F, ch.var->ntile > 0);   // (frame f: channel f, SNR f)
    const size_t nlen = (size_t)noise_len(*sys, L);
    const size_t n_eq = (size_t)sys->N * (sys->S - 1) * F;
    const size_t scratch_elems = (size_t)ch.lay.pad + sys->tail_tx + (size_t)sys->S * (sys->N + sys->cp + sys->cs - sys->tail_tx) + 64;
    const size_t scratch_bytes = ch.use_global ? (size_t)grid * 2 * scratch_elems * elem_bytes(*sys) : 0;

    rc = arena_reserve(h, d, t.bytes() + n_sym * 4 + nlen * F * 16 + n_eq * 16 + n_eq * 4 + (size_t)F * 16 + scratch_bytes);
    if (rc) return rc;
    void *d_wtx, *d_wrx, *d_tw, *d_chan, *d_snr, *d_sym, *d_noise, *d_eq, *d_dec, *d_be, *d_se, *d_scr = nullptr;
    WOFDM_CUDA(h, arena_put(d, t.wtx.data(), t.wtx.size(), &d_wtx));
    WOFDM_CUDA(h, arena_put(d, t.wrx.data(), t.wrx.size(), &d_wrx));
    WOFDM_CUDA(h, arena_put(d, t.tw.data(), t.tw.size(), &d_tw));
    WOFDM_CUDA(h, arena_put(d, t.chan.data(), t.chan.size(), &d_chan));
    WOFDM_CUDA(h, arena_put(d, t.snr.data(), t.snr.size(), &d_snr));
    WOFDM_CUDA(h, arena_put(d, sym_idx, n_sym * 4, &d_sym));
    WOFDM_CUDA(h, arena_put(d, noise, nlen * F * 16, &d_noise));
    WOFDM_CUDA(h, arena_put(d, nullptr, n_eq * 16, &d_eq));
    WOFDM_CUDA(h, arena_put(d, nullptr, n_eq * 4, &d_dec));
    WOFDM_CUDA(h, arena_put(d, nullptr, (size_t)F * 8, &d_be));
    WOFDM_CUDA(h, arena_put(d, nullptr, (size_t)F * 8, &d_se));
    if (scratch_bytes) WOFDM_CUDA(h, arena_put(d, nullptr, scratch_bytes, &d_scr));
    WOFDM_CUDA(h, cudaMemsetAsync(d_be, 0, (size_t)F * 8, d.stream));
    WOFDM_CUDA(h, cudaMemsetAsync(d_se, 0, (size_t)F * 8, d.stream));

    BerParams prm;
    fill_sys(prm, *sys, L);
    prm.chunk = ch.chunk; prm.use_global = ch.use_global;
    fill_flat(prm, *sys, win_tx, win_rx);
    fill_split(prm, *ch.var);
    prm.win_tx = d_wtx; prm.win_rx = d_wrx; prm.tw = d_tw; prm.chan = d_chan; prm.snr_lin = d_snr;
    prm.C = F; prm.n_snr = F; prm.ensemble = 1;
    prm.frame_begin = 0; prm.frame_step = 1; prm.n_frames = F;
    prm.sym_idx = static_cast<const int32_t*>(d_sym);
    prm.noise_in = static_cast<const double2*>(d_noise);
    prm.eq_out = static_cast<double2*>(d_eq);
    prm.dec_out = static_cast<int32_t*>(d_dec);
    prm.bit_err_f = static_cast<long long*>(d_be);
    prm.sym_err_f = static_cast<long long*>(d_se);
    prm.scratch = d_scr; prm.scratch_elems = (long long)scratch_elems;
    WOFDM_CUDA(h, ch.var->launch(prm, grid, ch.lay.bytes, d.stream));
    h->launches += 1;
    WOFDM_CUDA(h, cudaMemcpyAsync(eq_out, d_eq, n_eq * 16, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(dec_idx, d_dec, n_eq * 4, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(bit_err, d_be, (size_t)F * 8, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(sym_err, d_se, (size_t)F * 8, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
    return WOFDM_OK;
}

int wofdm_ber_draws(wofdm_handle h, const wofdm_sys_t* sys, int L, uint64_t seed, uint32_t variant,
                    const int64_t* frame_ids, int F, int32_t* sym_idx, double* noise) {
    NvtxRange nvtx_("wofdm_ber_draws");
    if (!h) return WOFDM_EINVAL;
    int rc = validate_sys(h, sys, L);
    if (rc) return rc;
    if (!frame_ids || !sym_idx || !noise || F < 1) return fail(h, WOFDM_EINVAL, "bad buffer");
    DeviceCtx& d = h->devs[0];
    WOFDM_CUDA(h, cudaSetDevice(d.dev));
    const size_t nlen = (size_t)noise_len(*sys, L);
    const size_t n_sym = (size_t)sys->N * sys->S * F;
    rc = arena_reserve(h, d, (size_t)F * 8 + n_sym * 4 + nlen * F * 16);
    if (rc) return rc;
    long long* d_ids = static_cast<long long*>(arena_take(d, (size_t)F * 8));
    int32_t* d_sym = static_cast<int32_t*>(arena_take(d, n_sym * 4));
    double2* d_noise = static_cast<double2*>(arena_take(d, nlen * F * 16));
    if (!d_ids || !d_sym || !d_noise) return fail(h, WOFDM_ENOMEM, "arena exhausted");
    WOFDM_CUDA(h, cudaMemcpyAsync(d_ids, frame_ids, (size_t)F * 8, cudaMemcpyHostToDevice, d.stream));
    BerParams prm;
    fill_sys(prm, *sys, L);
    prm.seed = seed; prm.variant = variant;
    philox_round_keys(seed, prm.rk);
    {   // the noise block B is a property of the kernel variant production mode dispatches to
        Choice ch;
        rc = choose_variant(h, *sys, L, d.smem_optin, KernelRequest{}, &ch);
        if (rc) return rc;
        prm.chunk = ch.chunk;
        fill_split(prm, *ch.var);
    }
    const dim3 gs(sys->S, F);
    switch (sys->N) {
        case 16: draws_sym_kernel<16><<<gs, 32, 0, d.stream>>>(prm, d_ids, d_sym); break;
        case 32: draws_sym_kernel<32><<<gs, 32, 0, d.stream>>>(prm, d_ids, d_sym); break;
        case 64: draws_sym_kernel<64><<<gs, 32, 0, d.stream>>>(prm, d_ids, d_sym); break;
        case 128: draws_sym_kernel<128><<<gs, 32, 0, d.stream>>>(prm, d_ids, d_sym); break;
        case 256: draws_sym_kernel<256><<<gs, 32, 0, d.stream>>>(prm, d_ids, d_sym); break;
        case 512: draws_sym_kernel<512><<<gs, 32, 0, d.stream>>>(prm, d_ids, d_sym); break;
        case 1024: draws_sym_kernel<1024><<<gs, 64, 0, d.stream>>>(prm, d_ids, d_sym); break;
        default: return fail(h, WOFDM_EUNSUPPORTED, "N");
    }
    WOFDM_CUDA(h, cudaGetLastError());
    const dim3 gn((unsigned)((nlen + 127) / 128), F);
    if (sys->precision == 1) draws_noise_kernel<double><<<gn, 128, 0, d.stream>>>(prm, d_ids, d_noise);
    else draws_noise_kernel<float><<<gn, 128, 0, d.stream>>>(prm, d_ids, d_noise);
    WOFDM_CUDA(h, cudaGetLastError());
    h->launches += 2;
    WOFDM_CUDA(h, cudaMemcpyAsync(sym_idx, d_sym, n_sym * 4, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaMemcpyAsync(noise, d_noise, nlen * F * 16, cudaMemcpyDeviceToHost, d.stream));
    WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
    return WOFDM_OK;
}

// in-place forward FFT of n = 2^k interleaved complex doubles (host; set-up of the mask response only)
static void host_fft_pow2(std::vector<double>& a, int n) {
    for (int i = 1, j = 0; i < n; ++i) {
        int bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) { std::swap(a[2 * i], a[2 * j]); std::swap(a[2 * i + 1], a[2 * j + 1]); }
    }
    for (int len = 2; len <= n; len <<= 1) {
        const double ang = -6.283185307179586476925286766559 / len;
        for (int i = 0; i < n; i += len)
            for (int k = 0; k < len / 2; ++k) {
                const double wr = std::cos(ang * k), wi = std::sin(ang * k);
                const int u = i + k, v = i + k + len / 2;
                const double xr = a[2 * v] * wr - a[2 * v + 1] * wi, xi = a[2 * v] * wi + a[2 * v + 1] * wr;
                a[2 * v] = a[2 * u] - xr; a[2 * v + 1] = a[2 * u + 1] - xi;
                a[2 * u] += xr; a[2 * u + 1] += xi;
            }
    }
}

}  // extern "C"

// Channel-mask variant (include/wofdm.h): frames in batches -- the masked Tx streams of a batch are written to HBM (the dense
// tensor-core product of mask_gemm.cu, or tx_mask_kernel with WOFDM_MASK_FFT=1), a K1 kernel reads them
// (BerParams::tx_stream) and does channel, noise, Rx and counting as always.
// A call is set up once (masked_setup: kernels, tables, device buffers, the mask product's matrices) and then runs ranges of
// frames (masked_run): global frame ids, or local indices of a segment table (wofdm_ber_run_masked_segments / _adaptive).
// n_var window pairs (wofdm_ber_run_masked_multi) share the batch's symbol draw and one product; K1 evaluates them in one
// launch where the gathering kernel holds all their tables, else one launch per pair.
namespace {

struct MaskedDev {
    int slot = 0;                          // device of the handle
    MaskGemm mg{};
    MaskParams mp{};                       // pair 0's; pair v: its Tx table and mask response (WOFDM_MASK_FFT=1)
    std::vector<BerParams> prm;            // one K1 launch each: all pairs, or pair v
    unsigned long long* d_cnt = nullptr;   // counter pairs [n_var][n_snr][Cr][Nr]
    void* d_stream = nullptr;
    long long* d_seg = nullptr;            // segment table [seg_cap][4]
};

struct MaskedJob {
    wofdm_ctx* h = nullptr;
    wofdm_sys_t sys{};
    Choice run;                            // the K1 kernel that runs
    bool use_gemm = false, fused = false;
    const char* dump_env = nullptr;
    long long max_ctas = 0, batch = 0, ensemble = 0;
    size_t ncnt = 0, cnt_bytes = 0, body = 0;   // (of one pair)
    int C = 0, seg_cap = 0, n_var = 1;
    std::vector<MaskedDev> devs;           // the devices set up: the first ones of the handle
};

// Set-up of a checked channel-mask call of n_var window pairs (win_tx / win_rx back to back, roll_off[n_var]; pair v's
// noise stream is variant + v): the kernels, the tables, and on every device that takes part (contiguous ranges of at least
// 64 frames out of max_frames, the most frames one masked_run covers) its buffers and the mask product's matrices.
// resolve != 0 or seg_cap > 0: the resolved twin of the K1 kernel (counters [n_var][n_snr][Cr][Nr], [n_var][n_snr] with
// resolve 0); seg_cap > 0 also gives every device a segment table of seg_cap entries.
int masked_setup(MaskedJob& J, wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                 const int* roll_off, const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                 uint64_t seed, uint32_t variant, int resolve, long long max_frames, int seg_cap) {
    const int N = sys->N, n_tx = N + sys->cp + sys->cs, stride = n_tx - sys->tail_tx, M = 2 * n_tx - 1, n_wr = N + sys->tail_rx;
    J.h = h; J.sys = *sys; J.C = C; J.ensemble = ensemble; J.seg_cap = seg_cap; J.n_var = n_var;
    const int Cr = (resolve & WOFDM_BY_CHANNEL) ? C : 1, Nr = (resolve & WOFDM_BY_SUBCARRIER) ? N : 1;
    J.ncnt = (size_t)n_snr * Cr * Nr;
    J.cnt_bytes = J.ncnt * 16;
    DeviceCtx& d0 = h->devs[0];              // (variant selection: the devices of a handle are alike)
    WOFDM_CUDA(h, cudaSetDevice(d0.dev));
    Choice ch;
    std::vector<Choice> prod(n_var);
    // Tx side: the dense tensor-core product of mask_gemm.cu; WOFDM_MASK_FFT=1 keeps the per-symbol FFT kernel (mask_kernel.cuh)
    const char* mask_env = getenv("WOFDM_MASK_FFT");
    J.use_gemm = !(mask_env && atoi(mask_env) == 1);
    J.dump_env = seg_cap > 0 ? nullptr : getenv("WOFDM_MASK_DUMP");     // (a development aid of the unsegmented calls)
    // a second-generation tensor-core kernel that gathers its stream from the product's output itself (no assembled copy in
    // HBM) where the frame fits one, else a tx_stream kernel (tuned or staged)
    int rc = WOFDM_OK;
    if (J.use_gemm && !(J.dump_env && *J.dump_env)) {
        KernelRequest rq;
        rq.no_circ = true;
        rq.tx = TxSource::gather;
        rc = choose_variant(h, *sys, L, d0.smem_optin, rq, &ch);
        J.fused = rc == WOFDM_OK && ch.var->txy;
    }
    if (!J.fused) {
        KernelRequest rq;
        rq.no_circ = true;
        rq.tx = TxSource::stream;
        rc = choose_variant(h, *sys, L, d0.smem_optin, rq, &ch);
    }
    if (rc) return rc;
    if (ch.var->CL > 1) return fail(h, WOFDM_EUNSUPPORTED, "no channel-mask variant for cluster kernels");
    for (int v = 0; v < n_var; ++v) {
        KernelRequest rq;                   // noise numbering of wofdm_ber_run / _draws with pair v's Tx window
        rq.win_tx = win_tx + (size_t)v * n_tx;
        rc = choose_variant(h, *sys, L, d0.smem_optin, rq, &prod[v]);
        if (rc) return rc;
        if (prod[v].var->CL > 1) return fail(h, WOFDM_EUNSUPPORTED, "no channel-mask variant for cluster kernels");
    }
    // the kernel that runs: ch, or (resolved counters, segments) its twin -- the noise numbering below stays ch's either way,
    // so a staged fallback draws ch's noise; it reads the assembled stream even where ch gathers from the product itself.
    // Several pairs: one launch of the gathering kernel (or of its twin) for all of them where it holds all their tables
    // and accumulators (the same kernel as for one pair, so the same counters); else one launch per pair on the shared
    // product output.
    int nv_launch = 1;
    J.run = ch;
    if (resolve || seg_cap > 0) {
        Choice nz = ch;
        if (ch.var->TC == 0) nz.chunk = prod[0].chunk;
        bool rfused = false;
        rc = choose_resolved(h, *sys, L, d0.smem_optin, nz, J.fused, n_var, &J.run, &rfused);
        if (rc) return rc;
        J.fused = J.run.var->txy;
        if (rfused) nv_launch = n_var;
    } else if (J.fused && n_var > 1) {
        const BerSmem lay = ch.var->layout(sys->S, stride, sys->tail_tx, sys->tail_rx, L, n_var, 0);
        if (lay.bytes <= d0.smem_optin) { nv_launch = n_var; J.run.lay = lay; }
    }
    const Choice& run = J.run;
    int nb = 0;
    rc = prepare_kernel(h, *run.var, run.lay.bytes, d0.sm_count, &nb, &J.max_ctas);
    if (rc) return rc;
    if (max_frames == 0) return WOFDM_OK;
    // the circular convolution (mod M) of an n_tx-sample symbol = a linear one with the periodic extension of g on
    // [-(n_tx-1), M-1]: Gp = FFT_P of that sequence laid out circularly in P = 8N >= 4 n_tx - 3 points, times 1/P
    // (WOFDM_MASK_FFT=1: [n_var][P], pair v's mask)
    const int P = 8 * N;
    std::vector<float> g(J.use_gemm ? 2 : 2 * (size_t)P * n_var, 0.f);
    std::vector<unsigned char> twp;
    for (int v = 0; v < n_var && !J.use_gemm; ++v) {
        const int ro = roll_off[v];
        // g = IDFT_M(ifftshift(windowRC)), main_channel_mask.m:404-412, 477-493
        std::vector<double> wrc(M, 0.0);
        {
            const int wl = M / 2, rest = M - wl - 2 * ro, zl = rest / 2;
            for (int i = 0; i < ro; ++i) {
                const double ax = -(ro + 1) / 2.0 + 1.0 + i;
                const double x = std::sin(1.5707963267948966 * (0.5 + ax / ro));
                wrc[zl + i] = x * x;
                wrc[zl + ro + wl + (ro - 1 - i)] = x * x;
            }
            for (int i = 0; i < wl; ++i) wrc[zl + ro + i] = 1.0;
        }
        std::vector<double> gd(2 * (size_t)M);
        std::vector<double> phc(M), phs(M);
        for (int i = 0; i < M; ++i) {
            const double a = 6.283185307179586476925286766559 * (double)i / (double)M;
            phc[i] = std::cos(a); phs[i] = std::sin(a);
        }
        for (int n = 0; n < M; ++n) {
            double re = 0.0, im = 0.0;
            int idx = 0;                                         // k n mod M
            for (int k = 0; k < M; ++k) {                        // ifftshift: shifted[k] = wrc[(k + M/2) mod M] (odd M: floor)
                const double w = wrc[(k + M / 2) % M];
                if (w != 0.0) { re += w * phc[idx]; im += w * phs[idx]; }
                idx += n;
                if (idx >= M) idx -= M;
            }
            gd[2 * n] = re / M; gd[2 * n + 1] = im / M;
        }
        std::vector<double> gc(2 * (size_t)P, 0.0);
        for (int mm = -(n_tx - 1); mm <= M - 1; ++mm) {
            const int gi = ((mm % M) + M) % M, ci = ((mm % P) + P) % P;
            gc[2 * ci] = gd[2 * gi]; gc[2 * ci + 1] = gd[2 * gi + 1];
        }
        host_fft_pow2(gc, P);
        for (size_t i = 0; i < gc.size(); ++i) g[2 * (size_t)P * v + i] = (float)(gc[i] / P);
    }
    if (!J.use_gemm) cast_any(false, build_twiddles(P), twp);
    else twp.resize(16);
    // (tx_mask_kernel shares the Tx window's table: a common factor of its stream)
    const HostTables t = build_tables(*sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, run.var->ntile > 0);
    J.body = (size_t)sys->tail_tx + (size_t)sys->S * stride;
    J.batch = std::min<long long>(max_frames, J.use_gemm ? 16384 : 8192);
    const size_t scratch_elems = (size_t)run.lay.pad + J.body + 64;
    const int grid_ber = (int)std::min<long long>(J.batch, J.max_ctas);
    const size_t scratch_bytes = run.use_global ? (size_t)grid_ber * 2 * scratch_elems * sizeof(float2) : 0;
    // every device of the handle takes a contiguous range of the frames (frame ids are global: same draws, same counters as
    // on one device); its work is enqueued on its own stream, the counters meet on the host
    const int nd = (int)std::min<long long>((long long)h->devs.size(), std::max<long long>(1, max_frames / 64));
    auto setup_dev = [&](MaskedDev& md) -> int {
        DeviceCtx& d = h->devs[md.slot];
        WOFDM_CUDA(h, cudaSetDevice(d.dev));
        if (&d != &d0) {
            int nb_ = 0; long long mc_ = 0;
            const int rcp = prepare_kernel(h, *run.var, run.lay.bytes, d.sm_count, &nb_, &mc_);
            if (rcp) return rcp;
        }
        const size_t mg_bytes = J.use_gemm ? mask_gemm_plan(*sys, J.batch, n_var, md.mg) : 0;
        const size_t stream_bytes = J.fused ? 16 : (size_t)J.batch * J.body * sizeof(float2);
        int rc = arena_reserve(h, d, t.bytes() + twp.size() + g.size() * 4 + n_var * J.cnt_bytes + stream_bytes + scratch_bytes +
                                     mg_bytes + (size_t)seg_cap * 32 + 8192);
        if (rc) return rc;
        void *d_wtx, *d_wrx, *d_tw, *d_twp, *d_chan, *d_snr, *d_g, *d_cnt, *d_seg = nullptr, *d_scr = nullptr;
        WOFDM_CUDA(h, arena_put(d, t.wtx.data(), t.wtx.size(), &d_wtx));
        WOFDM_CUDA(h, arena_put(d, t.wrx.data(), t.wrx.size(), &d_wrx));
        WOFDM_CUDA(h, arena_put(d, t.tw.data(), t.tw.size(), &d_tw));
        WOFDM_CUDA(h, arena_put(d, t.chan.data(), t.chan.size(), &d_chan));
        WOFDM_CUDA(h, arena_put(d, t.snr.data(), t.snr.size(), &d_snr));
        WOFDM_CUDA(h, arena_put(d, g.data(), g.size() * 4, &d_g));
        WOFDM_CUDA(h, arena_put(d, twp.data(), twp.size(), &d_twp));
        WOFDM_CUDA(h, arena_put(d, nullptr, n_var * J.cnt_bytes, &d_cnt));
        WOFDM_CUDA(h, arena_put(d, nullptr, stream_bytes, &md.d_stream));
        if (scratch_bytes) WOFDM_CUDA(h, arena_put(d, nullptr, scratch_bytes, &d_scr));
        if (seg_cap > 0) WOFDM_CUDA(h, arena_put(d, nullptr, (size_t)seg_cap * 32, &d_seg));
        md.d_cnt = static_cast<unsigned long long*>(d_cnt);
        md.d_seg = static_cast<long long*>(d_seg);
        if (J.use_gemm) {
            rc = mask_gemm_setup(h, d, md.mg, roll_off, static_cast<const float*>(d_wtx));
            if (rc) return rc;
        }
        MaskParams& mp = md.mp;
        memset(&mp, 0, sizeof(mp));
        mp.N = N; mp.cp = sys->cp; mp.cs = sys->cs; mp.tail_tx = sys->tail_tx; mp.bits = sys->bits; mp.S = sys->S;
        mp.n_tx = n_tx; mp.stride = stride; mp.constellation = sys->constellation; mp.guard = sys->guard; mp.M = M;
        mp.win_tx = static_cast<const float*>(d_wtx); mp.tw = static_cast<const float2*>(d_tw);
        mp.Gp = static_cast<const float2*>(d_g); mp.twp = static_cast<const float2*>(d_twp);
        mp.seed = seed; mp.stream = static_cast<float2*>(md.d_stream);
        // the K1 launches: pairs v .. v + nv_launch - 1 each (the tables, counters and product outputs of pair v on)
        md.prm.assign(n_var / nv_launch, BerParams{});
        for (int v = 0; v < n_var; v += nv_launch) {
            BerParams& prm = md.prm[v / nv_launch];
            fill_sys(prm, *sys, L);
            prm.chunk = ch.var->TC > 0 ? ch.chunk : prod[v].chunk; prm.use_global = run.use_global;
            fill_flat(prm, *sys, win_tx + (size_t)v * n_tx, win_rx + (size_t)v * n_wr, nv_launch);
            prm.flat_tx = 0;                       // (the Tx stream comes from tx_mask_kernel)
            prm.nvar = nv_launch;
            fill_split(prm, *ch.var);
            if (ch.var->TC == 0) {                 // staged kernel: the noise numbering of wofdm_ber_run / _draws (noise_at follows it)
                BerParams tmp = prm;
                fill_split(tmp, *prod[v].var);
                prm.n48 = tmp.n48;
            }
            prm.win_tx = static_cast<const float*>(d_wtx) + (size_t)v * n_tx;
            prm.win_rx = static_cast<const float*>(d_wrx) + (size_t)v * n_wr;
            prm.tw = d_tw; prm.chan = d_chan; prm.snr_lin = d_snr;
            prm.C = C; prm.n_snr = n_snr; prm.ensemble = ensemble; prm.seed = seed; prm.variant = variant + (uint32_t)v;
            philox_round_keys(seed, prm.rk);
            prm.counters = md.d_cnt + (size_t)v * J.ncnt * 2;
            prm.res_chan = (resolve & WOFDM_BY_CHANNEL) ? 1 : 0;
            prm.res_bins = (resolve & WOFDM_BY_SUBCARRIER) ? 1 : 0;
            prm.scratch = d_scr; prm.scratch_elems = (long long)scratch_elems;
            prm.tx_stream = static_cast<const float2*>(md.d_stream);
            if (J.fused) { prm.tx_y = md.mg.Y + (size_t)v * md.mg.ypair; prm.tx_yp = md.mg.Yp; prm.tx_ypair = md.mg.ypair; }
        }
        return WOFDM_OK;
    };
    J.devs.resize(nd);
    for (int i = 0; i < nd && rc == WOFDM_OK; ++i) {
        J.devs[i].slot = i;
        rc = setup_dev(J.devs[i]);
    }
    // (the host tables may go out of scope: uploads from pageable memory return once staged.  After a failure nothing of
    //  this call stays in flight.)
    if (rc)
        for (int i = 0; i < nd; ++i) { cudaSetDevice(h->devs[i].dev); cudaStreamSynchronize(h->devs[i].stream); }
    cudaSetDevice(d0.dev);
    return rc;
}

// The frames [g_lo, g_hi) of a set-up call: global frame ids, or with `segs` (at most seg_cap segments, its table uploaded to
// every device) local indices of that segment list.  The devices take contiguous ranges of at least 64.
// -> bit_err / sym_err [n_var][n_snr][Cr][Nr]
int masked_run(MaskedJob& J, long long g_lo, long long g_hi, const Segments* segs, int64_t* bit_err, int64_t* sym_err) {
    wofdm_ctx* h = J.h;
    const wofdm_sys_t& sys = J.sys;
    const int N = sys.N;
    const long long nfr = g_hi - g_lo;
    const size_t nout = (size_t)J.n_var * J.ncnt;
    if (nfr == 0) {
        for (size_t i = 0; i < nout; ++i) { bit_err[i] = 0; sym_err[i] = 0; }
        return WOFDM_OK;
    }
    const int n_seg = segs ? segs->n() : 0;
    if (n_seg > J.seg_cap) return fail(h, WOFDM_EINVAL, "more segments than the call's segment table holds");
    const int nd = (int)std::min<long long>((long long)J.devs.size(), std::max<long long>(1, nfr / 64));
    auto run_dev = [&](MaskedDev& md, long long f_lo, long long f_hi) -> int {
        DeviceCtx& d = h->devs[md.slot];
        WOFDM_CUDA(h, cudaSetDevice(d.dev));
        const long long* seg = segs ? md.d_seg : nullptr;
        // (pageable source: the copy returns once the table is staged; the previous work on this stream is ordered before it)
        if (segs) WOFDM_CUDA(h, cudaMemcpyAsync(md.d_seg, segs->tab.data(), segs->tab.size() * sizeof(long long), cudaMemcpyHostToDevice, d.stream));
        WOFDM_CUDA(h, cudaMemsetAsync(md.d_cnt, 0, J.n_var * J.cnt_bytes, d.stream));
        MaskSegParams mp;
        static_cast<MaskParams&>(mp) = md.mp;
        mp.seg = seg; mp.n_seg = n_seg; mp.C = J.C; mp.ensemble = J.ensemble;
        const int P = 8 * N, nvl = J.n_var / (int)md.prm.size();     // pairs per K1 launch
        for (long long f0 = f_lo; f0 < f_hi; f0 += J.batch) {
            const long long nf = std::min(J.batch, f_hi - f0);
            mp.frame_begin = f0; mp.frame_step = 1; mp.n_frames = nf;
            const int mgrid = (int)std::min<long long>(nf, (long long)d.sm_count);
            if (J.use_gemm) {      // every pair's masked symbols of the batch, one symbol draw and one product
                const int rc = mask_gemm_batch(h, d, md.mg, mp.seed, f0, nf, seg, n_seg, J.C, J.ensemble);
                if (rc) return rc;
            }
            for (size_t k = 0; k < md.prm.size(); ++k) {
                const int v = (int)k * nvl;                              // (first) pair of this K1 launch
                cudaError_t e = cudaSuccess;
                if (J.use_gemm) {
                    // the K1 kernel gathers from Y itself (ber_tconv2.cuh, tconv2_load_masked), or reads pair v's assembled stream
                    if (!J.fused) {
                        const int rc = mask_gemm_assemble(h, d, md.mg, v, nf, static_cast<float2*>(md.d_stream));
                        if (rc) return rc;
                    }
                } else {
                    mp.win_tx = md.mp.win_tx + (size_t)v * mp.n_tx;
                    mp.Gp = md.mp.Gp + (size_t)v * P;
                    // (SEG: the segmented instantiation, whose parameters carry the table)
                    auto launch = [&](auto kern_plain, auto kern_seg, size_t msm) {
                        cudaError_t es = cudaFuncSetAttribute(seg ? (const void*)kern_seg : (const void*)kern_plain,
                                                              cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm);
                        if (es == cudaSuccess && seg) kern_seg<<<mgrid, 256, msm, d.stream>>>(mp);
                        else if (es == cudaSuccess) kern_plain<<<mgrid, 256, msm, d.stream>>>(static_cast<const MaskParams&>(mp));
                        return es;
                    };
                    switch (N) {
                        case 128: e = launch(tx_mask_kernel<128>, tx_mask_kernel<128, true>, MaskSmem<128>::bytes(sys.S, mp.stride, sys.tail_tx)); break;
                        case 256: e = launch(tx_mask_kernel<256>, tx_mask_kernel<256, true>, MaskSmem<256>::bytes(sys.S, mp.stride, sys.tail_tx)); break;
                        default:  e = launch(tx_mask_kernel<512>, tx_mask_kernel<512, true>, MaskSmem<512>::bytes(sys.S, mp.stride, sys.tail_tx)); break;
                    }
                }
                WOFDM_CUDA(h, e);
                WOFDM_CUDA(h, cudaGetLastError());
                if (f0 == 0 && !segs && v == 0) {
                    // development aid: WOFDM_MASK_DUMP=<file> writes the masked Tx streams of the first (up to 4) frames as raw float32 pairs
                    const char* dump = J.dump_env;
                    if (dump && *dump) {
                        std::vector<float> hs(2 * J.body * (size_t)std::min<long long>(nf, 4));
                        WOFDM_CUDA(h, cudaMemcpyAsync(hs.data(), md.d_stream, hs.size() * 4, cudaMemcpyDeviceToHost, d.stream));
                        WOFDM_CUDA(h, cudaStreamSynchronize(d.stream));
                        if (FILE* fp = fopen(dump, "wb")) { fwrite(hs.data(), 4, hs.size(), fp); fclose(fp); }
                    }
                }
                BerParams prm = md.prm[k];
                prm.seg = seg; prm.n_seg = n_seg;
                prm.frame_begin = f0; prm.frame_step = 1; prm.n_frames = nf;
                WOFDM_CUDA(h, J.run.var->launch(prm, (int)std::min<long long>(nf, J.max_ctas), J.run.lay.bytes, d.stream));
                h->launches += 2;
            }
        }
        return WOFDM_OK;
    };
    int rc = WOFDM_OK;
    for (int i = 0; i < nd; ++i) {
        rc = run_dev(J.devs[i], g_lo + nfr * i / nd, g_lo + nfr * (i + 1) / nd);
        if (rc) break;
    }
    std::vector<std::vector<unsigned long long>> cnts;
    if (!rc) {
        try { cnts.assign(nd, std::vector<unsigned long long>(nout * 2, 0ull)); }
        catch (const std::bad_alloc&) { rc = fail(h, WOFDM_ENOMEM, "host allocation failed"); }
    }
    // (the downloads into pageable memory block the host: only after every device has its work)
    for (int i = 0; i < nd; ++i) {           // (also after a failure: nothing of this call stays in flight)
        DeviceCtx& d = h->devs[J.devs[i].slot];
        cudaSetDevice(d.dev);
        cudaError_t es = cudaSuccess;
        if (!rc) es = cudaMemcpyAsync(cnts[i].data(), J.devs[i].d_cnt, J.n_var * J.cnt_bytes, cudaMemcpyDeviceToHost, d.stream);
        if (es == cudaSuccess) es = cudaStreamSynchronize(d.stream);
        if (es != cudaSuccess && !rc) rc = fail(h, WOFDM_ECUDA, std::string("wofdm_ber_run_masked: ") + cudaGetErrorString(es));
    }
    cudaSetDevice(h->devs[0].dev);
    if (rc) return rc;
    for (size_t i = 0; i < nout; ++i) {
        unsigned long long be = 0, se = 0;
        for (int k = 0; k < nd; ++k) { be += cnts[k][2 * i]; se += cnts[k][2 * i + 1]; }
        bit_err[i] = (int64_t)be; sym_err[i] = (int64_t)se;
    }
    return WOFDM_OK;
}

// A checked job of the channel-mask chain for n_var window pairs: the whole job (segs == nullptr: global frame ids, the
// unsegmented kernels) or the frames of a segment list, in either case this shard's contiguous block of the local indices.
// resolve == 0: bit_err / sym_err [n_var][n_snr]; else [n_var][n_snr][Cr][Nr] (wofdm_ber_run_resolved's layout), counted by
// the resolved twin of the K1 kernel this chain picks.  Totals as in run_job; bit_tot may be NULL.
int run_masked_impl(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                    const int* roll_off, const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                    const Segments* segs, uint64_t seed, uint32_t variant, int shard_index, int shard_count, int resolve,
                    int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot, int64_t* bit_tot) {
    const Segments all = segs ? Segments() : job_segments(C, std::vector<int64_t>(n_snr, ensemble));
    const Segments& sg = segs ? *segs : all;
    const ShardRule r = ShardRule::block(sg.n_local, shard_index, shard_count);
    MaskedJob J;
    int rc = masked_setup(J, h, sys, win_tx, win_rx, n_var, roll_off, chan, L, C, snr_db, n_snr, ensemble, seed, variant, resolve,
                          r.hi - r.lo, segs ? segs->n() : 0);
    if (!rc) rc = masked_run(J, r.lo, r.hi, segs, bit_err, sym_err);
    if (rc) return rc;
    const int Cr = (resolve & WOFDM_BY_CHANNEL) ? C : 1, Nr = (resolve & WOFDM_BY_SUBCARRIER) ? sys->N : 1;
    cell_totals(*sys, cell_frames(sg, n_snr, C, Cr, r), Nr, sym_tot, bit_tot);
    return WOFDM_OK;
}

}  // namespace

extern "C" {

int wofdm_ber_run_masked(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                         uint64_t seed, uint32_t variant, int roll_off,
                         int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot) {
    return wofdm_ber_run_masked_shard(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble, seed, variant, roll_off, 0, 1,
                                      bit_err, bit_tot, sym_err, sym_tot);
}
int wofdm_ber_run_masked_shard(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                               const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                               uint64_t seed, uint32_t variant, int roll_off, int shard_index, int shard_count,
                               int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_masked");
    if (!h) return WOFDM_EINVAL;
    const int rc = check_masked(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble, roll_off, shard_index, shard_count, 0,
                                bit_err && bit_tot && sym_err && sym_tot);
    if (rc) return rc;
    return run_masked_impl(h, sys, win_tx, win_rx, 1, &roll_off, chan, L, C, snr_db, n_snr, ensemble, nullptr, seed, variant,
                           shard_index, shard_count, 0, bit_err, sym_err, sym_tot, bit_tot);
}

int wofdm_ber_run_masked_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                               const int* roll_off, int n_var, const double* chan, int L, int C, const double* snr_db, int n_snr,
                               int64_t ensemble, uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                               int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_masked_multi");
    if (!h) return WOFDM_EINVAL;
    const int rc = check_masked_multi(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble, roll_off, n_var, shard_index,
                                      shard_count, 0, bit_err && bit_tot && sym_err && sym_tot);
    if (rc) return rc;
    return run_masked_impl(h, sys, win_tx, win_rx, n_var, roll_off, chan, L, C, snr_db, n_snr, ensemble, nullptr, seed, variant,
                           shard_index, shard_count, 0, bit_err, sym_err, sym_tot, bit_tot);
}

int wofdm_ber_run_masked_resolved(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                                  const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                                  uint64_t seed, uint32_t variant, int roll_off, int shard_index, int shard_count, int resolve,
                                  int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_masked_resolved");
    if (!h) return WOFDM_EINVAL;
    int rc = check_resolve(h, resolve, true);
    if (rc) return rc;
    if (!bit_err || !sym_err || !sym_tot) return fail(h, WOFDM_EINVAL, "NULL output buffer");
    rc = check_masked(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble, roll_off, shard_index, shard_count, resolve, true);
    if (rc) return rc;
    return run_masked_impl(h, sys, win_tx, win_rx, 1, &roll_off, chan, L, C, snr_db, n_snr, ensemble, nullptr, seed, variant,
                           shard_index, shard_count, resolve, bit_err, sym_err, sym_tot, nullptr);
}

int wofdm_ber_run_masked_segments(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                                  const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                                  const int64_t* segments, int n_seg, uint64_t seed, uint32_t variant, int roll_off,
                                  int shard_index, int shard_count, int resolve, int64_t* bit_err, int64_t* sym_err,
                                  int64_t* sym_tot) {
    return wofdm_ber_run_masked_segments_multi(h, sys, win_tx, win_rx, &roll_off, 1, chan, L, C, snr_db, n_snr, ensemble_max,
                                               segments, n_seg, seed, variant, shard_index, shard_count, resolve, bit_err,
                                               sym_err, sym_tot);
}

int wofdm_ber_run_masked_segments_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                                        const int* roll_off, int n_var, const double* chan, int L, int C, const double* snr_db,
                                        int n_snr, int64_t ensemble_max, const int64_t* segments, int n_seg, uint64_t seed,
                                        uint32_t variant, int shard_index, int shard_count, int resolve, int64_t* bit_err,
                                        int64_t* sym_err, int64_t* sym_tot) {
    NvtxRange nvtx_("wofdm_ber_run_masked_segments");
    if (!h) return WOFDM_EINVAL;
    int rc = check_resolve(h, resolve, false);
    if (!rc) rc = check_masked_multi(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble_max, roll_off, n_var, shard_index,
                                     shard_count, resolve, bit_err && sym_err && sym_tot);
    if (!rc) rc = check_segments(h, segments, n_seg, n_snr, ensemble_max);
    if (rc) return rc;
    const Segments sg = seg_table(segments, n_seg, C);
    return run_masked_impl(h, sys, win_tx, win_rx, n_var, roll_off, chan, L, C, snr_db, n_snr, ensemble_max, &sg, seed, variant,
                           shard_index, shard_count, resolve, bit_err, sym_err, sym_tot, nullptr);
}

int wofdm_ber_run_masked_adaptive(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                                  const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                                  int64_t first_block, int target_kind, int64_t target, uint64_t seed, uint32_t variant,
                                  int roll_off, int shard_index, int shard_count, wofdm_reduce_fn reduce, void* reduce_user,
                                  int64_t* ensemble_used, int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot,
                                  int* rounds) {
    return wofdm_ber_run_masked_adaptive_multi(h, sys, win_tx, win_rx, &roll_off, 1, chan, L, C, snr_db, n_snr, ensemble_max,
                                               first_block, target_kind, target, seed, variant, shard_index, shard_count, reduce,
                                               reduce_user, ensemble_used, bit_err, bit_tot, sym_err, sym_tot, rounds);
}

int wofdm_ber_run_masked_adaptive_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                                        const int* roll_off, int n_var, const double* chan, int L, int C, const double* snr_db,
                                        int n_snr, int64_t ensemble_max, int64_t first_block, int target_kind, int64_t target,
                                        uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                                        wofdm_reduce_fn reduce, void* reduce_user, int64_t* ensemble_used, int64_t* bit_err,
                                        int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot, int* rounds) {
    NvtxRange nvtx_("wofdm_ber_run_masked_adaptive");
    if (!h) return WOFDM_EINVAL;
    const bool outputs_ok = ensemble_used && bit_err && bit_tot && sym_err && sym_tot && rounds;
    int rc = check_masked_multi(h, sys, win_tx, win_rx, chan, L, C, snr_db, n_snr, ensemble_max, roll_off, n_var, shard_index,
                                shard_count, 0, outputs_ok);
    if (!rc) rc = check_target(h, target_kind, target, first_block, shard_count, reduce);
    if (rc) return rc;
    if (variant > 0xfffffff0u - WOFDM_MAX_VARIANTS) return fail(h, WOFDM_EINVAL, "variant too large");
    // rows [0, n_var): the masked chain, pair v on noise stream variant + n_var + v, set up once for the largest round of
    // this shard; rows [n_var, 2 n_var): the unmasked chain, pair v on variant + v, a plan of its own device buffers (the
    // masked chain's live in the arena).  Each chain shards by its own rule.
    const long long total = (long long)n_snr * C * ensemble_max;
    const size_t half = (size_t)n_var * n_snr;
    MaskedJob J;
    rc = masked_setup(J, h, sys, win_tx, win_rx, n_var, roll_off, chan, L, C, snr_db, n_snr, ensemble_max, seed,
                      variant + (uint32_t)n_var, 0, (long long)(((__int128)total + shard_count - 1) / shard_count), n_snr);
    if (rc) return rc;
    wofdm_ber_plan p = nullptr;
    rc = plan_create_impl(h, sys, win_tx, win_rx, n_var, chan, L, C, snr_db, n_snr, &p, false, 0, n_snr);
    if (rc) return rc;
    rc = run_adaptive(h, *sys, C, n_snr, 2 * n_var, ensemble_max, first_block, target_kind, target, reduce, reduce_user,
                      [&](const Segments& sg, int64_t* be, int64_t* se) {
                          const ShardRule r = ShardRule::block(sg.n_local, shard_index, shard_count);
                          const int rc_m = masked_run(J, r.lo, r.hi, &sg, be, se);
                          if (rc_m) return rc_m;
                          return run_plan(p, ensemble_max, seed, variant, shard_index, shard_count, &sg, be + half, se + half);
                      },
                      ensemble_used, bit_err, bit_tot, sym_err, sym_tot, rounds);
    wofdm_ber_plan_destroy(p);
    return rc;
}

}  // extern "C"
