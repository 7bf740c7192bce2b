// wofdm_mex.cpp -- MATLAB MEX gateway over libwofdm.so (include/wofdm.h).  Pure argument marshalling.
//
//   ber = wofdm_mex('run_simulation', ensemble, symbolsPerTx, bitsPerSubcarrier, numSubcar, cpLength, ...
//                   csLength, windowTx, channel, snr, tailTx, tailRx, windowRx, prefixRemovalLength, ...
//                   circularShiftLength [, seed])
//       -- the positional arguments of run_simulation, matlab/main_BER_calculation.m:230-232.
//   berSNR = wofdm_mex('run_simulation_sweep', <the same 14 arguments> [, seed])
//       -- channel is now the whole C x L matrix (rows = realisations) and snr a vector: the triple loop of the
//          driver, matlab/main_BER_calculation.m:66-87 (for snr, for channel: ber = ber + run_simulation(...);
//          berSNR(snrIndex) = ber/numChannels), as ONE device job.  Returns n_snr x 1.
//   P   = wofdm_mex('calculate_interference', cpLength, typeOFDM, windowTx, windowRx, numSubcar, tailTx, ...
//                   tailRx, channels [, mode])
//       -- calculate_interference, matlab/main_interference_calculation.m:177-180; the values the reference
//          reads from settingsData.mat / the channel file inside the function are passed explicitly.
//   berSNR = wofdm_mex('run_simulation_sweep_multi', ...)   every window variant of a (system, CP) on the same bits, one job
//   berK = wofdm_mex('run_simulation_per_subcarrier', ...)  the same, BER per sub-carrier: n_snr x N x n_var
//   [berSNR, ensembleUsed] = wofdm_mex('run_simulation_adaptive', ...)  the same, each SNR point stopped at a bit-error target
//   [berMasked, ber] = wofdm_mex('run_sim_mc', ...)          run_sim_mc of matlab/main_channel_mask.m:334-337
//   [berMasked, ber] = wofdm_mex('run_sim_mc_per_subcarrier', ...)  the same, BER per sub-carrier: N x 1 each (0 on guard bins)
//   [berMasked, ber, ensembleUsed] = wofdm_mex('run_sim_mc_adaptive', ...)  run_sim_mc, each SNR point stopped at a bit-error target
//   [berMasked, ber] = wofdm_mex('run_sim_mc_multi', ...)    run_sim_mc for several window pairs / roll-offs on the same symbols
//   [psdMasked, psd] = wofdm_mex('psd_sim_mc', ...)         the Tx spectra of run_sim_mc's frames with and without the mask
//   [berMasked, ber, ensembleUsed] = wofdm_mex('run_sim_mc_multi_adaptive', ...)  run_sim_mc_adaptive for several configurations
//   [psdMasked, psd] = wofdm_mex('psd_sim_mc_multi', ...)   psd_sim_mc for several windows / roll-offs on the same frames
//   H = wofdm_mex('window_hessian', ...)                     quad_objective_tx / _rx of matlab/window_optimization.m:596-680
//   H = wofdm_mex('window_hessian_expected', ...), 'quad_objective_tx_expected', 'quad_objective_rx_expected'
//       -- the same, averaged over a channel set (C x L, rows = realisations) instead of built from one impulse response
//   channels = wofdm_mex('gen_channels', ...)                the stored channel sets' generator
//       (argument lists at the functions below)
// Windows arrive as dense diagonal matrices (or vectors); channels as rows = realisations.
#ifdef WOFDM_MEX_STUB
#include "mex_stub.h"
#else
#include "mex.h"
#endif
#include <string.h>

#include <vector>

#include "../include/wofdm.h"

static wofdm_handle g_handle = nullptr;

static void at_exit() {
    if (g_handle) wofdm_destroy(g_handle);
    g_handle = nullptr;
}

static wofdm_handle handle() {
    if (!g_handle) {
        if (wofdm_create(&g_handle, 0) != WOFDM_OK)
            mexErrMsgIdAndTxt("wofdm:nodevice", "wofdm_create failed: no CUDA device (this library has no CPU path)");
        mexAtExit(at_exit);
    }
    return g_handle;
}

static void check(int rc, const char* what) {
    if (rc != WOFDM_OK) mexErrMsgIdAndTxt("wofdm:error", "%s failed (%d): %s", what, rc, wofdm_last_error(g_handle));
}

// diagonal of a square matrix, or the vector itself
static std::vector<double> diag_of(const mxArray* a, size_t want) {
    const size_t m = mxGetM(a), n = mxGetN(a);
    const double* p = mxGetPr(a);
    std::vector<double> d(want);
    if (m == want && n == want) {
        for (size_t i = 0; i < want; ++i) d[i] = p[i * (want + 1)];
    } else if (m * n == want) {
        for (size_t i = 0; i < want; ++i) d[i] = p[i];
    } else {
        mexErrMsgIdAndTxt("wofdm:size", "window must be a %d x %d diagonal matrix or a vector of that length", (int)want, (int)want);
    }
    return d;
}

// MATLAB complex (split storage) -> interleaved (re, im)
static std::vector<double> interleave(const mxArray* a, size_t count, size_t stride, size_t offset) {
    const double *re = mxGetPr(a), *im = mxIsComplex(a) ? mxGetPi(a) : nullptr;
    std::vector<double> z(2 * count);
    for (size_t i = 0; i < count; ++i) {
        z[2 * i] = re[offset + i * stride];
        z[2 * i + 1] = im ? im[offset + i * stride] : 0.0;
    }
    return z;
}

// channels(channelIndex, :) (C x L, rows = realisations) -> column-major L x C complex
static std::vector<double> channel_rows(const mxArray* a, int* L, int* C) {
    const size_t c_n = mxGetM(a), l_n = mxGetN(a);
    std::vector<double> chan(2 * l_n * c_n);
    for (size_t c = 0; c < c_n; ++c) {
        const std::vector<double> row = interleave(a, l_n, c_n, c);
        memcpy(chan.data() + 2 * l_n * c, row.data(), 2 * l_n * sizeof(double));
    }
    *L = (int)l_n;
    *C = (int)c_n;
    return chan;
}

// sweep = false: one channel (vector), one SNR -> scalar; sweep = true: C x L channel matrix, SNR vector -> n_snr x 1
static void do_run_simulation(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[], bool sweep) {
    if (nrhs < 14) mexErrMsgIdAndTxt("wofdm:nargin", "run_simulation needs 14 arguments");
    (void)nlhs;
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long ensemble = (long long)mxGetScalar(prhs[0]);
    s.S = (int)mxGetScalar(prhs[1]);
    s.bits = (int)mxGetScalar(prhs[2]);
    s.N = (int)mxGetScalar(prhs[3]);
    s.cp = (int)mxGetScalar(prhs[4]);
    s.cs = (int)mxGetScalar(prhs[5]);
    s.tail_tx = (int)mxGetScalar(prhs[9]);
    s.tail_rx = (int)mxGetScalar(prhs[10]);
    s.rm = (int)mxGetScalar(prhs[12]);
    s.shift = (int)mxGetScalar(prhs[13]);
    s.noise_norm = 1;      // add_wgn on the full convolution, main_BER_calculation.m:260,277-294
    s.constellation = 1;   // qammod(..., 'UnitAveragePower', true), :248
    s.precision = 0;
    const std::vector<double> wtx = diag_of(prhs[6], (size_t)(s.N + s.cp + s.cs));
    const std::vector<double> wrx = diag_of(prhs[11], (size_t)(s.N + s.tail_rx));
    const unsigned long long seed = nrhs > 14 ? (unsigned long long)mxGetScalar(prhs[14]) : 0ull;
    if (!sweep) {
        const int L = (int)mxGetNumberOfElements(prhs[7]);
        const std::vector<double> chan = interleave(prhs[7], (size_t)L, 1, 0);
        const double snr = mxGetScalar(prhs[8]);
        long long be = 0, bt = 0, se = 0, st = 0;
        check(wofdm_ber_run(handle(), &s, wtx.data(), wrx.data(), chan.data(), L, 1, &snr, 1, ensemble, seed, 0,
                            (int64_t*)&be, (int64_t*)&bt, (int64_t*)&se, (int64_t*)&st), "wofdm_ber_run");
        plhs[0] = mxCreateDoubleScalar(bt ? (double)be / (double)bt : 0.0);   // ber, as [~, ber] = biterr(...) at :272
        return;
    }
    // channels(channelIndex, :) -> column-major L x C complex
    const size_t C = mxGetM(prhs[7]), L = mxGetN(prhs[7]);
    std::vector<double> chan(2 * L * C);
    for (size_t c = 0; c < C; ++c) {
        const std::vector<double> row = interleave(prhs[7], L, C, c);
        memcpy(chan.data() + 2 * L * c, row.data(), 2 * L * sizeof(double));
    }
    const size_t n_snr = mxGetNumberOfElements(prhs[8]);
    const double* snr = mxGetPr(prhs[8]);
    std::vector<long long> be(n_snr), bt(n_snr), se(n_snr), st(n_snr);
    check(wofdm_ber_run(handle(), &s, wtx.data(), wrx.data(), chan.data(), (int)L, (int)C, snr, (int)n_snr, ensemble, seed, 0,
                        (int64_t*)be.data(), (int64_t*)bt.data(), (int64_t*)se.data(), (int64_t*)st.data()), "wofdm_ber_run");
    plhs[0] = mxCreateDoubleMatrix((mwSize)n_snr, 1, mxREAL);
    double* out = mxGetPr(plhs[0]);
    for (size_t i = 0; i < n_snr; ++i) out[i] = bt[i] ? (double)be[i] / (double)bt[i] : 0.0;
}

// {w1, w2, ...} (cell array of diagonal matrices / vectors) or one window -> n_var windows back to back
static std::vector<double> windows_of(const mxArray* a, size_t want, size_t* n_var) {
    std::vector<double> all;
    if (mxIsCell(a)) {
        *n_var = mxGetNumberOfElements(a);
        for (size_t v = 0; v < *n_var; ++v) {
            const std::vector<double> w = diag_of(mxGetCell(a, v), want);
            all.insert(all.end(), w.begin(), w.end());
        }
    } else {
        *n_var = 1;
        all = diag_of(a, want);
    }
    return all;
}

// berSNR = wofdm_mex('run_simulation_sweep_multi', <the 14 arguments of run_simulation_sweep> [, seed]) with windowTx and
// windowRx CELL ARRAYS of n_var windows (a single window is repeated): every window pair on the same bits, one device job
// -- the {optimised, RC} pairs of matlab/main_BER_calculation.m:66-117 and the RC + CaseA/CaseB steps 1-3 of :118-198.
// Returns n_snr x n_var; column v = run_simulation_sweep with pair v (its noise stream: variant v).
// per_subcarrier = true ('run_simulation_per_subcarrier', the same arguments): BER of every sub-carrier,
// n_snr x N x n_var (FFT bin order; guard bins 0), from wofdm_ber_run_resolved on the same draws.
// adaptive = true ('run_simulation_adaptive', the 14 arguments, then targetBitErrors, ensembleMax [, seed]): every SNR point
// runs until each pair has counted targetBitErrors bit errors or ensembleMax ensemble indices (wofdm_ber_run_adaptive);
// the first argument, ensemble, is the first round's block.  Returns [berSNR (n_snr x n_var), ensembleUsed (n_snr x 1)].
static void do_run_simulation_multi(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[], bool per_subcarrier,
                                    bool adaptive = false) {
    const char* name = adaptive ? "run_simulation_adaptive" : per_subcarrier ? "run_simulation_per_subcarrier" : "run_simulation_sweep_multi";
    if (nrhs < (adaptive ? 16 : 14)) mexErrMsgIdAndTxt("wofdm:nargin", "%s needs %d arguments", name, adaptive ? 16 : 14);
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long ensemble = (long long)mxGetScalar(prhs[0]);
    s.S = (int)mxGetScalar(prhs[1]); s.bits = (int)mxGetScalar(prhs[2]); s.N = (int)mxGetScalar(prhs[3]);
    s.cp = (int)mxGetScalar(prhs[4]); s.cs = (int)mxGetScalar(prhs[5]);
    s.tail_tx = (int)mxGetScalar(prhs[9]); s.tail_rx = (int)mxGetScalar(prhs[10]);
    s.rm = (int)mxGetScalar(prhs[12]); s.shift = (int)mxGetScalar(prhs[13]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    const size_t n_tx = (size_t)(s.N + s.cp + s.cs), n_wr = (size_t)(s.N + s.tail_rx);
    size_t nvt = 0, nvr = 0;
    std::vector<double> wtx = windows_of(prhs[6], n_tx, &nvt), wrx = windows_of(prhs[11], n_wr, &nvr);
    const size_t n_var = nvt > nvr ? nvt : nvr;
    if ((nvt != n_var && nvt != 1) || (nvr != n_var && nvr != 1) || n_var > WOFDM_MAX_VARIANTS)
        mexErrMsgIdAndTxt("wofdm:size", "windowTx / windowRx: cell arrays of the same length (<= %d), or one window", WOFDM_MAX_VARIANTS);
    while (wtx.size() < n_var * n_tx) wtx.insert(wtx.end(), wtx.begin(), wtx.begin() + n_tx);
    while (wrx.size() < n_var * n_wr) wrx.insert(wrx.end(), wrx.begin(), wrx.begin() + n_wr);
    const int seed_arg = adaptive ? 16 : 14;
    const unsigned long long seed = nrhs > seed_arg ? (unsigned long long)mxGetScalar(prhs[seed_arg]) : 0ull;
    const size_t C = mxGetM(prhs[7]), L = mxGetN(prhs[7]);
    std::vector<double> chan(2 * L * C);
    for (size_t c = 0; c < C; ++c) {
        const std::vector<double> row = interleave(prhs[7], L, C, c);
        memcpy(chan.data() + 2 * L * c, row.data(), 2 * L * sizeof(double));
    }
    const size_t n_snr = mxGetNumberOfElements(prhs[8]);
    if (per_subcarrier) {
        const size_t N = (size_t)s.N;
        std::vector<long long> be(n_var * n_snr * N), se(n_var * n_snr * N), st(n_snr * N);
        check(wofdm_ber_run_resolved(handle(), &s, wtx.data(), wrx.data(), (int)n_var, chan.data(), (int)L, (int)C, mxGetPr(prhs[8]),
                                     (int)n_snr, ensemble, seed, 0, 0, 1, WOFDM_BY_SUBCARRIER, (int64_t*)be.data(), (int64_t*)se.data(),
                                     (int64_t*)st.data()),
              "wofdm_ber_run_resolved");
        const mwSize dims[3] = {(mwSize)n_snr, (mwSize)N, (mwSize)n_var};
        plhs[0] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);
        double* out = mxGetPr(plhs[0]);
        for (size_t v = 0; v < n_var; ++v)          // column-major: out(i, k, v)
            for (size_t k = 0; k < N; ++k)
                for (size_t i = 0; i < n_snr; ++i) {
                    const long long bt = st[i * N + k] * s.bits;
                    out[(v * N + k) * n_snr + i] = bt ? (double)be[(v * n_snr + i) * N + k] / (double)bt : 0.0;
                }
        return;
    }
    std::vector<long long> be(n_var * n_snr), se(n_var * n_snr), bt(n_snr), st(n_snr);
    if (adaptive) {
        std::vector<long long> used(n_snr);
        int rounds = 0;
        check(wofdm_ber_run_adaptive(handle(), &s, wtx.data(), wrx.data(), (int)n_var, chan.data(), (int)L, (int)C, mxGetPr(prhs[8]),
                                     (int)n_snr, (long long)mxGetScalar(prhs[15]), ensemble, WOFDM_TARGET_BIT_ERRORS,
                                     (long long)mxGetScalar(prhs[14]), seed, 0, 0, 1, nullptr, nullptr, (int64_t*)used.data(),
                                     (int64_t*)be.data(), (int64_t*)bt.data(), (int64_t*)se.data(), (int64_t*)st.data(), &rounds),
              "wofdm_ber_run_adaptive");
        plhs[0] = mxCreateDoubleMatrix((mwSize)n_snr, (mwSize)n_var, mxREAL);
        double* out = mxGetPr(plhs[0]);
        for (size_t v = 0; v < n_var; ++v)
            for (size_t i = 0; i < n_snr; ++i) out[v * n_snr + i] = bt[i] ? (double)be[v * n_snr + i] / (double)bt[i] : 0.0;
        if (nlhs > 1) {
            plhs[1] = mxCreateDoubleMatrix((mwSize)n_snr, 1, mxREAL);
            for (size_t i = 0; i < n_snr; ++i) mxGetPr(plhs[1])[i] = (double)used[i];
        }
        return;
    }
    check(wofdm_ber_run_multi(handle(), &s, wtx.data(), wrx.data(), (int)n_var, chan.data(), (int)L, (int)C, mxGetPr(prhs[8]), (int)n_snr,
                              ensemble, seed, 0, 0, 1, (int64_t*)be.data(), (int64_t*)bt.data(), (int64_t*)se.data(), (int64_t*)st.data()),
          "wofdm_ber_run_multi");
    plhs[0] = mxCreateDoubleMatrix((mwSize)n_snr, (mwSize)n_var, mxREAL);
    double* out = mxGetPr(plhs[0]);
    for (size_t v = 0; v < n_var; ++v)
        for (size_t i = 0; i < n_snr; ++i) out[v * n_snr + i] = bt[i] ? (double)be[v * n_snr + i] / (double)bt[i] : 0.0;
}

// [berMasked, ber] = wofdm_mex('run_sim_mc', ensemble, cpLength, csLength, tailTx, tailRx, windowTx, windowRx, channel, snr,
//                               offset, prefixRemovalLength, circularShiftLength, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff [, seed])
//   -- the positional arguments of run_sim_mc, matlab/main_channel_mask.m:334-337: the same symbols with and without the
//      DFT-domain raised-cosine mask, independent noise, averaged over the ensemble.
// per_subcarrier = true ('run_sim_mc_per_subcarrier', the same arguments): berMasked and ber of every sub-carrier, N x 1 in
// FFT bin order, 0 on the guard bins; their mean over the active bins is run_sim_mc's result.
static void do_run_sim_mc(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[], bool per_subcarrier) {
    const char* name = per_subcarrier ? "run_sim_mc_per_subcarrier" : "run_sim_mc";
    if (nrhs < 16) mexErrMsgIdAndTxt("wofdm:nargin", "%s needs 16 arguments", name);
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long ensemble = (long long)mxGetScalar(prhs[0]);
    s.cp = (int)mxGetScalar(prhs[1]); s.cs = (int)mxGetScalar(prhs[2]);
    s.tail_tx = (int)mxGetScalar(prhs[3]); s.tail_rx = (int)mxGetScalar(prhs[4]);
    s.guard = (int)mxGetScalar(prhs[9]); s.rm = (int)mxGetScalar(prhs[10]); s.shift = (int)mxGetScalar(prhs[11]);
    s.N = (int)mxGetScalar(prhs[12]); s.bits = (int)mxGetScalar(prhs[13]); s.S = (int)mxGetScalar(prhs[14]);
    const int roll_off = (int)mxGetScalar(prhs[15]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    const std::vector<double> wtx = diag_of(prhs[5], (size_t)(s.N + s.cp + s.cs));
    const std::vector<double> wrx = diag_of(prhs[6], (size_t)(s.N + s.tail_rx));
    const int L = (int)mxGetNumberOfElements(prhs[7]);
    const std::vector<double> chan = interleave(prhs[7], (size_t)L, 1, 0);
    const double snr = mxGetScalar(prhs[8]);
    const unsigned long long seed = nrhs > 16 ? (unsigned long long)mxGetScalar(prhs[16]) : 0ull;
    if (per_subcarrier) {
        const size_t N = (size_t)s.N;
        std::vector<long long> be(N), se(N), st(N), bem(N), sem(N), stm(N);
        check(wofdm_ber_run_resolved(handle(), &s, wtx.data(), wrx.data(), 1, chan.data(), L, 1, &snr, 1, ensemble, seed, 0, 0, 1,
                                     WOFDM_BY_SUBCARRIER, (int64_t*)be.data(), (int64_t*)se.data(), (int64_t*)st.data()),
              "wofdm_ber_run_resolved");
        check(wofdm_ber_run_masked_resolved(handle(), &s, wtx.data(), wrx.data(), chan.data(), L, 1, &snr, 1, ensemble, seed, 1,
                                            roll_off, 0, 1, WOFDM_BY_SUBCARRIER, (int64_t*)bem.data(), (int64_t*)sem.data(),
                                            (int64_t*)stm.data()),
              "wofdm_ber_run_masked_resolved");
        plhs[0] = mxCreateDoubleMatrix((mwSize)N, 1, mxREAL);
        double* om = mxGetPr(plhs[0]);
        for (size_t k = 0; k < N; ++k) om[k] = stm[k] ? (double)bem[k] / (double)(stm[k] * s.bits) : 0.0;
        if (nlhs > 1) {
            plhs[1] = mxCreateDoubleMatrix((mwSize)N, 1, mxREAL);
            double* o = mxGetPr(plhs[1]);
            for (size_t k = 0; k < N; ++k) o[k] = st[k] ? (double)be[k] / (double)(st[k] * s.bits) : 0.0;
        }
        return;
    }
    long long be = 0, bt = 0, se = 0, st = 0, bem = 0, btm = 0;
    check(wofdm_ber_run(handle(), &s, wtx.data(), wrx.data(), chan.data(), L, 1, &snr, 1, ensemble, seed, 0,
                        (int64_t*)&be, (int64_t*)&bt, (int64_t*)&se, (int64_t*)&st), "wofdm_ber_run");
    check(wofdm_ber_run_masked(handle(), &s, wtx.data(), wrx.data(), chan.data(), L, 1, &snr, 1, ensemble, seed, 1, roll_off,
                               (int64_t*)&bem, (int64_t*)&btm, (int64_t*)&se, (int64_t*)&st), "wofdm_ber_run_masked");
    plhs[0] = mxCreateDoubleScalar(btm ? (double)bem / (double)btm : 0.0);
    if (nlhs > 1) plhs[1] = mxCreateDoubleScalar(bt ? (double)be / (double)bt : 0.0);
}

// [berMasked, ber] = wofdm_mex('run_sim_mc_multi', <the 16 arguments of run_sim_mc> [, seed]) with windowTx and windowRx CELL
// ARRAYS of n_var windows and rollOff a vector of n_var, channel C x L (rows = realisations) and snr a vector
//   -- every configuration v = (windowTx{v}, windowRx{v}, rollOff(v)) on the same symbols: the unmasked chain in one call
//      (wofdm_ber_run_multi, noise stream v), the masked chain in one (wofdm_ber_run_masked_multi, noise stream n_var + v).
//      Each output is n_snr x n_var.
static void do_run_sim_mc_multi(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 16) mexErrMsgIdAndTxt("wofdm:nargin", "run_sim_mc_multi needs 16 arguments");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long ensemble = (long long)mxGetScalar(prhs[0]);
    s.cp = (int)mxGetScalar(prhs[1]); s.cs = (int)mxGetScalar(prhs[2]);
    s.tail_tx = (int)mxGetScalar(prhs[3]); s.tail_rx = (int)mxGetScalar(prhs[4]);
    s.guard = (int)mxGetScalar(prhs[9]); s.rm = (int)mxGetScalar(prhs[10]); s.shift = (int)mxGetScalar(prhs[11]);
    s.N = (int)mxGetScalar(prhs[12]); s.bits = (int)mxGetScalar(prhs[13]); s.S = (int)mxGetScalar(prhs[14]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    size_t nvt = 0, nvr = 0;
    const std::vector<double> wtx = windows_of(prhs[5], (size_t)(s.N + s.cp + s.cs), &nvt);
    const std::vector<double> wrx = windows_of(prhs[6], (size_t)(s.N + s.tail_rx), &nvr);
    const size_t n_var = mxGetNumberOfElements(prhs[15]);
    if (nvt != n_var || nvr != n_var || n_var < 1 || n_var > WOFDM_MAX_VARIANTS)
        mexErrMsgIdAndTxt("wofdm:size", "windowTx, windowRx (cell arrays) and rollOff must all hold n_var <= %d entries", WOFDM_MAX_VARIANTS);
    std::vector<int> roll_off(n_var);
    for (size_t v = 0; v < n_var; ++v) roll_off[v] = (int)mxGetPr(prhs[15])[v];
    int L = 0, C = 0;
    const std::vector<double> chan = channel_rows(prhs[7], &L, &C);
    const size_t n_snr = mxGetNumberOfElements(prhs[8]);
    const unsigned long long seed = nrhs > 16 ? (unsigned long long)mxGetScalar(prhs[16]) : 0ull;
    std::vector<long long> be(n_var * n_snr), se(n_var * n_snr), bt(n_snr), st(n_snr), bem(n_var * n_snr), sem(n_var * n_snr), btm(n_snr);
    check(wofdm_ber_run_multi(handle(), &s, wtx.data(), wrx.data(), (int)n_var, chan.data(), L, C, mxGetPr(prhs[8]), (int)n_snr,
                              ensemble, seed, 0, 0, 1, (int64_t*)be.data(), (int64_t*)bt.data(), (int64_t*)se.data(), (int64_t*)st.data()),
          "wofdm_ber_run_multi");
    check(wofdm_ber_run_masked_multi(handle(), &s, wtx.data(), wrx.data(), roll_off.data(), (int)n_var, chan.data(), L, C,
                                     mxGetPr(prhs[8]), (int)n_snr, ensemble, seed, (uint32_t)n_var, 0, 1, (int64_t*)bem.data(),
                                     (int64_t*)btm.data(), (int64_t*)sem.data(), (int64_t*)st.data()),
          "wofdm_ber_run_masked_multi");
    for (int row = 0; row < 2 && row < (nlhs > 0 ? nlhs : 1); ++row) {      // berMasked, ber
        const std::vector<long long>& e = row == 0 ? bem : be;
        const std::vector<long long>& t = row == 0 ? btm : bt;
        plhs[row] = mxCreateDoubleMatrix((mwSize)n_snr, (mwSize)n_var, mxREAL);
        double* out = mxGetPr(plhs[row]);
        for (size_t v = 0; v < n_var; ++v)
            for (size_t i = 0; i < n_snr; ++i) out[v * n_snr + i] = t[i] ? (double)e[v * n_snr + i] / (double)t[i] : 0.0;
    }
}

// [berMasked, ber, ensembleUsed] = wofdm_mex('run_sim_mc_adaptive', <the 16 arguments of run_sim_mc>, targetBitErrors,
//                                            ensembleMax [, seed])
//   -- run_sim_mc with every SNR point stopped once the masked and the unmasked chain have each counted targetBitErrors
//      bit errors, or at ensembleMax ensemble indices (wofdm_ber_run_masked_adaptive).  channel: C x L (rows = realisations),
//      snr: a vector; the first argument, ensemble, is the first round's block.  Each output is n_snr x 1.
static void do_run_sim_mc_adaptive(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 18) mexErrMsgIdAndTxt("wofdm:nargin", "run_sim_mc_adaptive needs 18 arguments");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long first_block = (long long)mxGetScalar(prhs[0]);
    s.cp = (int)mxGetScalar(prhs[1]); s.cs = (int)mxGetScalar(prhs[2]);
    s.tail_tx = (int)mxGetScalar(prhs[3]); s.tail_rx = (int)mxGetScalar(prhs[4]);
    s.guard = (int)mxGetScalar(prhs[9]); s.rm = (int)mxGetScalar(prhs[10]); s.shift = (int)mxGetScalar(prhs[11]);
    s.N = (int)mxGetScalar(prhs[12]); s.bits = (int)mxGetScalar(prhs[13]); s.S = (int)mxGetScalar(prhs[14]);
    const int roll_off = (int)mxGetScalar(prhs[15]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    const std::vector<double> wtx = diag_of(prhs[5], (size_t)(s.N + s.cp + s.cs));
    const std::vector<double> wrx = diag_of(prhs[6], (size_t)(s.N + s.tail_rx));
    const size_t C = mxGetM(prhs[7]), L = mxGetN(prhs[7]);
    std::vector<double> chan(2 * L * C);
    for (size_t c = 0; c < C; ++c) {
        const std::vector<double> row = interleave(prhs[7], L, C, c);
        memcpy(chan.data() + 2 * L * c, row.data(), 2 * L * sizeof(double));
    }
    const size_t n_snr = mxGetNumberOfElements(prhs[8]);
    const long long target = (long long)mxGetScalar(prhs[16]), ensemble_max = (long long)mxGetScalar(prhs[17]);
    const unsigned long long seed = nrhs > 18 ? (unsigned long long)mxGetScalar(prhs[18]) : 0ull;
    std::vector<long long> be(2 * n_snr), se(2 * n_snr), bt(n_snr), st(n_snr), used(n_snr);
    int rounds = 0;
    check(wofdm_ber_run_masked_adaptive(handle(), &s, wtx.data(), wrx.data(), chan.data(), (int)L, (int)C, mxGetPr(prhs[8]),
                                        (int)n_snr, ensemble_max, first_block, WOFDM_TARGET_BIT_ERRORS, target, seed, 0, roll_off,
                                        0, 1, nullptr, nullptr, (int64_t*)used.data(), (int64_t*)be.data(), (int64_t*)bt.data(),
                                        (int64_t*)se.data(), (int64_t*)st.data(), &rounds),
          "wofdm_ber_run_masked_adaptive");
    for (int row = 0; row < 3 && row < (nlhs > 0 ? nlhs : 1); ++row) {       // berMasked (row 0), ber (row 1), ensembleUsed
        plhs[row] = mxCreateDoubleMatrix((mwSize)n_snr, 1, mxREAL);
        double* out = mxGetPr(plhs[row]);
        for (size_t i = 0; i < n_snr; ++i)
            out[i] = row == 2 ? (double)used[i] : bt[i] ? (double)be[row * n_snr + i] / (double)bt[i] : 0.0;
    }
}

// [berMasked, ber, ensembleUsed] = wofdm_mex('run_sim_mc_multi_adaptive', <the 16 arguments of run_sim_mc_multi>,
//                                            targetBitErrors, ensembleMax [, seed])
//   -- run_sim_mc_adaptive for every configuration v = (windowTx{v}, windowRx{v}, rollOff(v)) on the same symbols in one
//      call (wofdm_ber_run_masked_adaptive_multi): the noise streams of run_sim_mc_multi, every SNR point stopped once all
//      2 n_var chains have counted targetBitErrors bit errors, or at ensembleMax.  The first argument is the first round's
//      block.  berMasked and ber are n_snr x n_var, ensembleUsed n_snr x 1.
static void do_run_sim_mc_multi_adaptive(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 18) mexErrMsgIdAndTxt("wofdm:nargin", "run_sim_mc_multi_adaptive needs 18 arguments");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long first_block = (long long)mxGetScalar(prhs[0]);
    s.cp = (int)mxGetScalar(prhs[1]); s.cs = (int)mxGetScalar(prhs[2]);
    s.tail_tx = (int)mxGetScalar(prhs[3]); s.tail_rx = (int)mxGetScalar(prhs[4]);
    s.guard = (int)mxGetScalar(prhs[9]); s.rm = (int)mxGetScalar(prhs[10]); s.shift = (int)mxGetScalar(prhs[11]);
    s.N = (int)mxGetScalar(prhs[12]); s.bits = (int)mxGetScalar(prhs[13]); s.S = (int)mxGetScalar(prhs[14]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    size_t nvt = 0, nvr = 0;
    const std::vector<double> wtx = windows_of(prhs[5], (size_t)(s.N + s.cp + s.cs), &nvt);
    const std::vector<double> wrx = windows_of(prhs[6], (size_t)(s.N + s.tail_rx), &nvr);
    const size_t n_var = mxGetNumberOfElements(prhs[15]);
    if (nvt != n_var || nvr != n_var || n_var < 1 || n_var > WOFDM_MAX_VARIANTS)
        mexErrMsgIdAndTxt("wofdm:size", "windowTx, windowRx (cell arrays) and rollOff must all hold n_var <= %d entries", WOFDM_MAX_VARIANTS);
    std::vector<int> roll_off(n_var);
    for (size_t v = 0; v < n_var; ++v) roll_off[v] = (int)mxGetPr(prhs[15])[v];
    int L = 0, C = 0;
    const std::vector<double> chan = channel_rows(prhs[7], &L, &C);
    const size_t n_snr = mxGetNumberOfElements(prhs[8]);
    const long long target = (long long)mxGetScalar(prhs[16]), ensemble_max = (long long)mxGetScalar(prhs[17]);
    const unsigned long long seed = nrhs > 18 ? (unsigned long long)mxGetScalar(prhs[18]) : 0ull;
    std::vector<long long> be(2 * n_var * n_snr), se(2 * n_var * n_snr), bt(n_snr), st(n_snr), used(n_snr);
    int rounds = 0;
    check(wofdm_ber_run_masked_adaptive_multi(handle(), &s, wtx.data(), wrx.data(), roll_off.data(), (int)n_var, chan.data(), L,
                                              C, mxGetPr(prhs[8]), (int)n_snr, ensemble_max, first_block,
                                              WOFDM_TARGET_BIT_ERRORS, target, seed, 0, 0, 1, nullptr, nullptr,
                                              (int64_t*)used.data(), (int64_t*)be.data(), (int64_t*)bt.data(),
                                              (int64_t*)se.data(), (int64_t*)st.data(), &rounds),
          "wofdm_ber_run_masked_adaptive_multi");
    for (int row = 0; row < 3 && row < (nlhs > 0 ? nlhs : 1); ++row) {       // berMasked (block 0), ber (block 1), ensembleUsed
        plhs[row] = mxCreateDoubleMatrix((mwSize)n_snr, row == 2 ? 1 : (mwSize)n_var, mxREAL);
        double* out = mxGetPr(plhs[row]);
        if (row == 2) {
            for (size_t i = 0; i < n_snr; ++i) out[i] = (double)used[i];
            continue;
        }
        for (size_t v = 0; v < n_var; ++v)
            for (size_t i = 0; i < n_snr; ++i)
                out[v * n_snr + i] = bt[i] ? (double)be[(row * n_var + v) * n_snr + i] / (double)bt[i] : 0.0;
    }
}

// H = wofdm_mex('window_hessian', typeOFDM, numSubcar, cpLength, tailTx, tailRx, channel)
//   -- the quadratic form of the interference power (ICI + ISI) in the REDUCED window variables (tail coefficients), as
//      python's OptimizerTx/Rx/TxRx.gen_hessian builds it.  channel: ONE impulse response.  (quad_objective_tx / _rx of
//      matlab/window_optimization.m:596-680 work in the full window variable with the other window fixed, weight the
//      two terms with alpha and keep only the diagonal of the ISI term: 'quad_objective_tx' / 'quad_objective_rx' below.)
// H = wofdm_mex('window_hessian_expected', typeOFDM, numSubcar, cpLength, tailTx, tailRx, channels)
//   -- the same averaged over the channel set (C x L, rows = realisations): the expected interference over the set.
static void do_window_hessian(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[], bool expected) {
    if (nrhs < 6) mexErrMsgIdAndTxt("wofdm:nargin", "window_hessian needs 6 arguments");
    (void)nlhs;
    char name[16];
    if (!mxIsChar(prhs[0]) || mxGetString(prhs[0], name, sizeof(name))) mexErrMsgIdAndTxt("wofdm:type", "typeOFDM must be a string");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    s.bits = 4; s.S = 2; s.precision = 1;
    if (wofdm_params_from_name(name, (int)mxGetScalar(prhs[1]), (int)mxGetScalar(prhs[2]), (int)mxGetScalar(prhs[3]),
                               (int)mxGetScalar(prhs[4]), &s) != WOFDM_OK)
        mexErrMsgIdAndTxt("wofdm:type", "unknown typeOFDM '%s'", name);
    const int n_var = (s.tail_rx / 2 + 1) * (s.tail_tx + 1);
    plhs[0] = mxCreateDoubleMatrix((mwSize)n_var, (mwSize)n_var, mxREAL);
    int nv = 0;
    if (expected) {
        int L = 0, C = 0;
        const std::vector<double> chan = channel_rows(prhs[5], &L, &C);
        check(wofdm_window_hessian_set(handle(), &s, chan.data(), L, C, mxGetPr(plhs[0]), &nv), "wofdm_window_hessian_set");
        return;
    }
    const int L = (int)mxGetNumberOfElements(prhs[5]);
    const std::vector<double> chan = interleave(prhs[5], (size_t)L, 1, 0);
    check(wofdm_window_hessian(handle(), &s, chan.data(), L, mxGetPr(plhs[0]), &nv), "wofdm_window_hessian");
}

// HTx = wofdm_mex('quad_objective_tx', typeOFDM, numSubcar, cpLength, tailTx, tailRx, windowRx, channel, alpha)
// HRx = wofdm_mex('quad_objective_rx', typeOFDM, numSubcar, cpLength, tailTx, tailRx, windowTx, channel, alpha)
//   -- quad_objective_tx / _rx of matlab/window_optimization.m:596-680: the FULL window of one side is the variable
//      (n_tx, or N + tailRx, entries), the other side's window (diagonal matrix or vector) is fixed:
//      H = 2 (alpha H1 + (1 - alpha) H2), H1 the off-diagonal ICI term, H2 = real(diag(diag(.))) of the ISI term (:628-631).
//      channel: ONE impulse response (the script passes array_ici_isi of the mean channel; the device builds those matrices).
// HTx = wofdm_mex('quad_objective_tx_expected', <the same arguments with channels C x L, rows = realisations>), and _rx:
//      the mean over the set of quad_objective_tx / _rx (the formula is linear in the two parts, so their means suffice).
static void do_quad_objective(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[], bool tx_side, bool expected) {
    if (nrhs < 8) mexErrMsgIdAndTxt("wofdm:nargin", "quad_objective_tx / _rx need 8 arguments");
    (void)nlhs;
    char name[16];
    if (!mxIsChar(prhs[0]) || mxGetString(prhs[0], name, sizeof(name))) mexErrMsgIdAndTxt("wofdm:type", "typeOFDM must be a string");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    s.bits = 4; s.S = 2; s.precision = 1;
    if (wofdm_params_from_name(name, (int)mxGetScalar(prhs[1]), (int)mxGetScalar(prhs[2]), (int)mxGetScalar(prhs[3]),
                               (int)mxGetScalar(prhs[4]), &s) != WOFDM_OK)
        mexErrMsgIdAndTxt("wofdm:type", "unknown typeOFDM '%s'", name);
    const size_t n_tx = (size_t)(s.N + s.cp + s.cs), n_w = (size_t)(s.N + s.tail_rx);
    const size_t n = tx_side ? n_tx : n_w;                       // variables: the full window of this side
    const std::vector<double> fixed = diag_of(prhs[5], tx_side ? n_w : n_tx);
    const double alpha = mxGetScalar(prhs[7]);
    std::vector<double> eye(n * n, 0.0), hc(n * n), hs(n * n);
    for (size_t i = 0; i < n; ++i) eye[i * n + i] = 1.0;
    const double* bt = tx_side ? eye.data() : fixed.data();
    const double* br = tx_side ? fixed.data() : eye.data();
    const int n_tb = tx_side ? (int)n : 1, n_rb = tx_side ? 1 : (int)n;
    if (expected) {
        int L = 0, C = 0;
        const std::vector<double> chan = channel_rows(prhs[6], &L, &C);
        check(wofdm_window_hessian_parts_set(handle(), &s, chan.data(), L, C, bt, n_tb, br, n_rb, hc.data(), hs.data()),
              "wofdm_window_hessian_parts_set");
    } else {
        const int L = (int)mxGetNumberOfElements(prhs[6]);
        const std::vector<double> chan = interleave(prhs[6], (size_t)L, 1, 0);
        check(wofdm_window_hessian_parts(handle(), &s, chan.data(), L, bt, n_tb, br, n_rb, hc.data(), hs.data()),
              "wofdm_window_hessian_parts");
    }
    plhs[0] = mxCreateDoubleMatrix((mwSize)n, (mwSize)n, mxREAL);
    double* H = mxGetPr(plhs[0]);
    for (size_t i = 0; i < n; ++i) {
        double row = 0.0;
        for (size_t j = 0; j < n; ++j) { row += hs[i * n + j]; H[i + j * n] = alpha * hc[i * n + j]; }
        H[i + i * n] += (1.0 - alpha) * row;
    }
}

// channels = wofdm_mex('gen_channels', standard, numTaps, dopplerFreq, samplingRate, frameDuration, noFrames, nSets [, seed])
//   -- ITU-R tapped-delay-line channels with GMEDS_1 fading (python/channel_model/itur_channels.py:33-94), the producer of the
//      stored channel sets; rows = realisations (set-major), as vehA200channel2(channelIndex, :) is indexed.
static void do_gen_channels(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 7) mexErrMsgIdAndTxt("wofdm:nargin", "gen_channels needs 7 arguments");
    (void)nlhs;
    char name[32];
    if (!mxIsChar(prhs[0]) || mxGetString(prhs[0], name, sizeof(name))) mexErrMsgIdAndTxt("wofdm:type", "standard must be a string");
    const int prof = wofdm_channel_profile(name);
    if (prof < 0) mexErrMsgIdAndTxt("wofdm:type", "unknown channel standard '%s'", name);
    const int L = (int)mxGetScalar(prhs[1]), no_frames = (int)mxGetScalar(prhs[5]), n_sets = (int)mxGetScalar(prhs[6]);
    const unsigned long long seed = nrhs > 7 ? (unsigned long long)mxGetScalar(prhs[7]) : 0ull;
    const size_t C = (size_t)no_frames * (size_t)n_sets;
    std::vector<double> chan(2 * (size_t)L * C);
    check(wofdm_gen_channels(handle(), prof, L, mxGetScalar(prhs[2]), mxGetScalar(prhs[3]), mxGetScalar(prhs[4]), no_frames, n_sets,
                             seed, nullptr, chan.data()), "wofdm_gen_channels");
    plhs[0] = mxCreateDoubleMatrix((mwSize)C, (mwSize)L, mxCOMPLEX);
    double *re = mxGetPr(plhs[0]), *im = mxGetPi(plhs[0]);
    for (size_t c = 0; c < C; ++c)
        for (int l = 0; l < L; ++l) { re[(size_t)l * C + c] = chan[2 * (c * L + l)]; im[(size_t)l * C + c] = chan[2 * (c * L + l) + 1]; }
}

static void do_calculate_interference(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 8) mexErrMsgIdAndTxt("wofdm:nargin", "calculate_interference needs 8 arguments");
    (void)nlhs;
    char name[16];
    if (!mxIsChar(prhs[1]) || mxGetString(prhs[1], name, sizeof(name))) mexErrMsgIdAndTxt("wofdm:type", "typeOFDM must be a string");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    s.bits = 4; s.S = 2; s.precision = 1;
    if (wofdm_params_from_name(name, (int)mxGetScalar(prhs[4]), (int)mxGetScalar(prhs[0]), (int)mxGetScalar(prhs[5]),
                               (int)mxGetScalar(prhs[6]), &s) != WOFDM_OK)
        mexErrMsgIdAndTxt("wofdm:type", "unknown typeOFDM '%s'", name);
    const std::vector<double> wtx = diag_of(prhs[2], (size_t)(s.N + s.cp + s.cs));
    const std::vector<double> wrx = diag_of(prhs[3], (size_t)(s.N + s.tail_rx));
    // channels: rows = realisations (vehA200channel2(channelIndex, :)); the reference uses their mean (:196)
    const size_t C = mxGetM(prhs[7]), L = mxGetN(prhs[7]);
    std::vector<double> mean(2 * L, 0.0);
    for (size_t c = 0; c < C; ++c) {
        const std::vector<double> row = interleave(prhs[7], L, C, c);
        for (size_t i = 0; i < 2 * L; ++i) mean[i] += row[i] / (double)C;
    }
    const int mode = nrhs > 8 ? (int)mxGetScalar(prhs[8]) : 0;
    double P = 0.0;
    check(wofdm_interf_power_scalar(handle(), &s, wtx.data(), wrx.data(), mean.data(), (int)L, 1, mode, &P),
          "wofdm_interf_power_scalar");
    plhs[0] = mxCreateDoubleScalar(P);
}

// [psdMasked, psd] = wofdm_mex('psd_sim_mc', numFrames, cpLength, csLength, tailTx, windowTx, offset, numSubcar,
//                               bitsPerSubcar, symbolsPerTx, rollOff [, seed [, estimator]])
//   -- the 8N-point fftshifted PSD (8N x 1 each) of the Tx signal of run_sim_mc's frames 0 .. numFrames-1 (the symbols
//      run_sim_mc draws with the same seed), with and without the DFT-domain raised-cosine mask (wofdm_psd_masked).
//      estimator: 'reference' / 0 (__psd_estimate's slices, the default) or 'hann' / 1 (sin^2 taper, 50 % overlap).
static void do_psd_sim_mc(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 10) mexErrMsgIdAndTxt("wofdm:nargin", "psd_sim_mc needs 10 arguments");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long n_frames = (long long)mxGetScalar(prhs[0]);
    s.cp = (int)mxGetScalar(prhs[1]); s.cs = (int)mxGetScalar(prhs[2]); s.tail_tx = (int)mxGetScalar(prhs[3]);
    s.guard = (int)mxGetScalar(prhs[5]); s.N = (int)mxGetScalar(prhs[6]); s.bits = (int)mxGetScalar(prhs[7]);
    s.S = (int)mxGetScalar(prhs[8]);
    const int roll_off = (int)mxGetScalar(prhs[9]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    const std::vector<double> wtx = diag_of(prhs[4], (size_t)(s.N + s.cp + s.cs));
    const unsigned long long seed = nrhs > 10 ? (unsigned long long)mxGetScalar(prhs[10]) : 0ull;
    int estimator = 0;
    if (nrhs > 11) {
        char est[16];
        if (mxIsChar(prhs[11])) {
            if (mxGetString(prhs[11], est, sizeof(est))) mexErrMsgIdAndTxt("wofdm:usage", "estimator: 'reference' or 'hann'");
            if (!strcmp(est, "hann")) estimator = 1;
            else if (strcmp(est, "reference")) mexErrMsgIdAndTxt("wofdm:usage", "estimator: 'reference' or 'hann'");
        } else {
            estimator = (int)mxGetScalar(prhs[11]);
        }
    }
    const size_t P = 8 * (size_t)(s.N > 0 ? s.N : 0);
    std::vector<double> xm(P), xu(P);
    check(wofdm_psd_masked(handle(), &s, wtx.data(), roll_off, seed, 0, n_frames, estimator, xm.data(), xu.data()),
          "wofdm_psd_masked");
    for (int k = 0; k < 2 && k < (nlhs > 0 ? nlhs : 1); ++k) {
        plhs[k] = mxCreateDoubleMatrix((mwSize)P, 1, mxREAL);
        memcpy(mxGetPr(plhs[k]), (k == 0 ? xm : xu).data(), P * sizeof(double));
    }
}

// [psdMasked, psd] = wofdm_mex('psd_sim_mc_multi', <the arguments of psd_sim_mc>) with windowTx a CELL ARRAY of n_var
// windows and rollOff a vector of n_var (or one value for every window)
//   -- psd_sim_mc for every configuration v = (windowTx{v}, rollOff(v)) on the same frames in one call
//      (wofdm_psd_masked_multi: the symbols drawn once, one mask product for all spectra).  Each output is 8N x n_var.
static void do_psd_sim_mc_multi(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 10) mexErrMsgIdAndTxt("wofdm:nargin", "psd_sim_mc_multi needs 10 arguments");
    wofdm_sys_t s;
    memset(&s, 0, sizeof(s));
    const long long n_frames = (long long)mxGetScalar(prhs[0]);
    s.cp = (int)mxGetScalar(prhs[1]); s.cs = (int)mxGetScalar(prhs[2]); s.tail_tx = (int)mxGetScalar(prhs[3]);
    s.guard = (int)mxGetScalar(prhs[5]); s.N = (int)mxGetScalar(prhs[6]); s.bits = (int)mxGetScalar(prhs[7]);
    s.S = (int)mxGetScalar(prhs[8]);
    s.noise_norm = 1; s.constellation = 1; s.precision = 0;
    size_t n_var = 0;
    const std::vector<double> wtx = windows_of(prhs[4], (size_t)(s.N + s.cp + s.cs), &n_var);
    const size_t n_ro = mxGetNumberOfElements(prhs[9]);
    if (n_var < 1 || n_var > WOFDM_MAX_VARIANTS || (n_ro != n_var && n_ro != 1))
        mexErrMsgIdAndTxt("wofdm:size", "windowTx (a cell array) must hold n_var <= %d windows and rollOff n_var values or one", WOFDM_MAX_VARIANTS);
    std::vector<int> roll_off(n_var);
    for (size_t v = 0; v < n_var; ++v) roll_off[v] = (int)mxGetPr(prhs[9])[n_ro == 1 ? 0 : v];
    const unsigned long long seed = nrhs > 10 ? (unsigned long long)mxGetScalar(prhs[10]) : 0ull;
    int estimator = 0;
    if (nrhs > 11) {
        char est[16];
        if (mxIsChar(prhs[11])) {
            if (mxGetString(prhs[11], est, sizeof(est))) mexErrMsgIdAndTxt("wofdm:usage", "estimator: 'reference' or 'hann'");
            if (!strcmp(est, "hann")) estimator = 1;
            else if (strcmp(est, "reference")) mexErrMsgIdAndTxt("wofdm:usage", "estimator: 'reference' or 'hann'");
        } else {
            estimator = (int)mxGetScalar(prhs[11]);
        }
    }
    const size_t P = 8 * (size_t)(s.N > 0 ? s.N : 0);
    std::vector<double> xm(P * n_var), xu(P * n_var);
    check(wofdm_psd_masked_multi(handle(), &s, wtx.data(), roll_off.data(), (int)n_var, seed, 0, n_frames, estimator, xm.data(),
                                 xu.data()),
          "wofdm_psd_masked_multi");
    for (int k = 0; k < 2 && k < (nlhs > 0 ? nlhs : 1); ++k) {       // column v = configuration v (row v of the library's output)
        plhs[k] = mxCreateDoubleMatrix((mwSize)P, (mwSize)n_var, mxREAL);
        memcpy(mxGetPr(plhs[k]), (k == 0 ? xm : xu).data(), P * n_var * sizeof(double));
    }
}

extern "C" void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    char cmd[32];
    if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], cmd, sizeof(cmd)))
        mexErrMsgIdAndTxt("wofdm:usage", "first argument: 'run_simulation', 'run_simulation_sweep', 'run_simulation_sweep_multi', 'run_simulation_per_subcarrier', 'run_simulation_adaptive', 'run_sim_mc', 'run_sim_mc_per_subcarrier', 'run_sim_mc_adaptive', 'run_sim_mc_multi', 'run_sim_mc_multi_adaptive', 'psd_sim_mc', 'psd_sim_mc_multi', 'calculate_interference', 'window_hessian', 'quad_objective_tx', 'quad_objective_rx', 'window_hessian_expected', 'quad_objective_tx_expected', 'quad_objective_rx_expected' or 'gen_channels'");
    if (!strcmp(cmd, "run_simulation")) do_run_simulation(nlhs, plhs, nrhs - 1, prhs + 1, false);
    else if (!strcmp(cmd, "run_simulation_sweep")) do_run_simulation(nlhs, plhs, nrhs - 1, prhs + 1, true);
    else if (!strcmp(cmd, "run_simulation_sweep_multi")) do_run_simulation_multi(nlhs, plhs, nrhs - 1, prhs + 1, false);
    else if (!strcmp(cmd, "run_simulation_per_subcarrier")) do_run_simulation_multi(nlhs, plhs, nrhs - 1, prhs + 1, true);
    else if (!strcmp(cmd, "run_simulation_adaptive")) do_run_simulation_multi(nlhs, plhs, nrhs - 1, prhs + 1, false, true);
    else if (!strcmp(cmd, "run_sim_mc")) do_run_sim_mc(nlhs, plhs, nrhs - 1, prhs + 1, false);
    else if (!strcmp(cmd, "run_sim_mc_per_subcarrier")) do_run_sim_mc(nlhs, plhs, nrhs - 1, prhs + 1, true);
    else if (!strcmp(cmd, "run_sim_mc_adaptive")) do_run_sim_mc_adaptive(nlhs, plhs, nrhs - 1, prhs + 1);
    else if (!strcmp(cmd, "run_sim_mc_multi")) do_run_sim_mc_multi(nlhs, plhs, nrhs - 1, prhs + 1);
    else if (!strcmp(cmd, "psd_sim_mc")) do_psd_sim_mc(nlhs, plhs, nrhs - 1, prhs + 1);
    else if (!strcmp(cmd, "run_sim_mc_multi_adaptive")) do_run_sim_mc_multi_adaptive(nlhs, plhs, nrhs - 1, prhs + 1);
    else if (!strcmp(cmd, "psd_sim_mc_multi")) do_psd_sim_mc_multi(nlhs, plhs, nrhs - 1, prhs + 1);
    else if (!strcmp(cmd, "window_hessian")) do_window_hessian(nlhs, plhs, nrhs - 1, prhs + 1, false);
    else if (!strcmp(cmd, "quad_objective_tx")) do_quad_objective(nlhs, plhs, nrhs - 1, prhs + 1, true, false);
    else if (!strcmp(cmd, "quad_objective_rx")) do_quad_objective(nlhs, plhs, nrhs - 1, prhs + 1, false, false);
    else if (!strcmp(cmd, "window_hessian_expected")) do_window_hessian(nlhs, plhs, nrhs - 1, prhs + 1, true);
    else if (!strcmp(cmd, "quad_objective_tx_expected")) do_quad_objective(nlhs, plhs, nrhs - 1, prhs + 1, true, true);
    else if (!strcmp(cmd, "quad_objective_rx_expected")) do_quad_objective(nlhs, plhs, nrhs - 1, prhs + 1, false, true);
    else if (!strcmp(cmd, "gen_channels")) do_gen_channels(nlhs, plhs, nrhs - 1, prhs + 1);
    else if (!strcmp(cmd, "calculate_interference")) do_calculate_interference(nlhs, plhs, nrhs - 1, prhs + 1);
    else mexErrMsgIdAndTxt("wofdm:usage", "unknown command '%s'", cmd);
}
