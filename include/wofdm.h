/* wofdm.h -- C-ABI of libwofdm.so, the B200-native replacement for the Monte-Carlo BER/SER
 * chain and the interference-power evaluation of felipescoelho/w-ofdm-optimization.
 *
 * The reference has no FFI: its boundary is function level.  Each entry point below names the
 * reference function it replaces (paths relative to the reference root).  Bindings: ctypes
 * (w-ofdm-optimization_b200/capi.py) for python/ofdm_utils, MEX gateway (mex/wofdm_mex.cpp) for
 * matlab/main_BER_calculation.m and matlab/main_interference_calculation.m; see INTEGRATION.md.
 *
 * Conventions: plain C, host pointers unless a parameter is named d_*; the caller owns every
 * buffer; complex = interleaved (re,im) doubles; matrices are column-major where MATLAB passes
 * matrices; every function returns 0 or a negative WOFDM_E* code and never throws; a handle is
 * not thread-safe, different handles are.  There is no CPU fallback: without a CUDA device
 * wofdm_create fails with WOFDM_ENODEV.
 */
#ifndef WOFDM_H_
#define WOFDM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WOFDM_VERSION 100

#if defined(__GNUC__)
#define WOFDM_API __attribute__((visibility("default")))
#else
#define WOFDM_API
#endif

enum {
    WOFDM_OK = 0,
    WOFDM_EINVAL = -1,       /* bad argument (see wofdm_last_error) */
    WOFDM_ECUDA = -2,        /* CUDA runtime error */
    WOFDM_ENOMEM = -3,       /* host or device allocation failed */
    WOFDM_ENODEV = -4,       /* no usable CUDA device */
    WOFDM_EUNSUPPORTED = -5  /* valid request outside the compiled kernel set */
};

typedef struct wofdm_ctx* wofdm_handle;
typedef struct wofdm_ber_plan_s* wofdm_ber_plan;

/* One w-OFDM system (SURVEY.md App. A.1).  n_tx = N+cp+cs, stride = n_rx = N+tail_rx+rm = n_tx-tail_tx. */
typedef struct {
    int32_t N;             /* DFT length, power of two in [16, 1024] */
    int32_t cp;            /* cyclic prefix */
    int32_t cs;            /* cyclic suffix */
    int32_t tail_tx;       /* Tx window tail */
    int32_t tail_rx;       /* Rx window tail (even) */
    int32_t rm;            /* samples dropped in front of each Rx block */
    int32_t shift;         /* circular shift before the DFT */
    int32_t bits;          /* bits per sub-carrier: 2, 4, 6 or 8 (square QAM) */
    int32_t S;             /* OFDM symbols per frame; symbol 0 is the pilot */
    int32_t noise_norm;    /* 0 = python: SNR fixed on the truncated signal (wofdm_simulation.py:208-215)
                              1 = matlab: on the full convolution (main_BER_calculation.m:260-261) */
    int32_t constellation; /* 0 = python: natural-order un-normalised list (wofdm_simulation.py:179-182)
                              1 = matlab: qammod Gray, unit average power (main_BER_calculation.m:248) */
    int32_t precision;     /* 0 = fp32, 1 = fp64 */
    int32_t guard;         /* null sub-carriers on EACH side of the centred spectrum (0 = all N carry data):
                              matlab/main_channel_mask.m:55,388-391 (`offset`, zeros + ifftshift).  FFT bin k is
                              active iff guard <= (k + N/2) mod N < N - guard; only active bins are counted.
                              Needs bits < 8. */
} wofdm_sys_t;

/* ---- library / device ------------------------------------------------------------------- */
WOFDM_API int wofdm_version(void);
WOFDM_API int wofdm_device_count(int* n);
/* n_gpus = 0: every visible device; n > 0: devices 0..n-1. */
WOFDM_API int wofdm_create(wofdm_handle* h, int n_gpus);
/* Explicit device list (one process per GPU under torchrun: {LOCAL_RANK}). */
WOFDM_API int wofdm_create_on(wofdm_handle* h, const int* device_ids, int n);
WOFDM_API int wofdm_destroy(wofdm_handle h);
WOFDM_API const char* wofdm_last_error(wofdm_handle h);
/* Kernels of this library launched through the handle so far. */
WOFDM_API int64_t wofdm_launch_count(wofdm_handle h);

/* Diagnostic: FMA-only micro-benchmark on device slot 0 (mode 0 scalar FFMA, 1 packed FFMA2).
 * tflops = measured FP32 rate, the denominator of the BER kernel's roofline; sm_mhz_equiv (optional)
 * = the SM clock at which 128 FMA lanes per SM would deliver that rate. */
WOFDM_API int wofdm_diag_fp32_peak(wofdm_handle h, int mode, double* tflops, double* sm_mhz_equiv);

/* ---- parameter table and windows (host, tiny) -------------------------------------------- */
/* Replaces wOFDMSystem.__init__'s table (python/ofdm_utils/wofdm_simulation.py:391-418) and
 * calculate_parameters (matlab/main_BER_calculation.m:457-493).  name: CP, wtx, CPwtx, wrx, CPwrx,
 * WOLA, CPW.  Fills N, cp, cs, tail_tx, tail_rx, rm, shift; leaves the other fields alone. */
WOFDM_API int wofdm_params_from_name(const char* name, int N, int cp, int tail_tx, int tail_rx, wofdm_sys_t* out);
/* gen_rc_window_tx / gen_rc_window_rx (python/ofdm_utils/transmitter.py:61-87, receiver.py:36-56;
 * matlab/functions/transmitter_rc_window.m, receiver_rc_window.m).  out: n_tx resp. N+tail_rx. */
WOFDM_API int wofdm_rc_window_tx(const wofdm_sys_t* sys, double* out);
WOFDM_API int wofdm_rc_window_rx(const wofdm_sys_t* sys, double* out);
/* reduce_variable_tx/rx applied to a stored tail vector (python/optimization_tools/utils.py:13-73):
 * x has tail_tx+1 resp. tail_rx/2+1 entries. */
WOFDM_API int wofdm_expand_window_tx(const wofdm_sys_t* sys, const double* x, double* out);
WOFDM_API int wofdm_expand_window_rx(const wofdm_sys_t* sys, const double* x, double* out);

/* ---- Monte-Carlo BER/SER chain ----------------------------------------------------------- */
/* Replaces wOFDMSystem.__run_sim_mc / __run_sim_cp_mc (python/ofdm_utils/wofdm_simulation.py:85-366)
 * and run_simulation (matlab/main_BER_calculation.m:230-274) for ONE window pair.  On-device Philox
 * draws.  Frames are indexed f = (snr_idx*C + chan_idx)*ensemble + e; symbols depend on (seed, f),
 * noise on (seed, f, variant): calling twice with the same seed and variant 0/1 evaluates two window
 * pairs on the same symbols with independent noise, as the reference does for optimised vs RC.
 * Counters are summed over channels x ensemble, one entry per SNR point; *_tot are the totals
 * (frames * N*bits*(S-1) resp. frames * N*(S-1)).  Uses every device of the handle.
 *   win_tx: n_tx doubles, win_rx: N+tail_rx doubles, chan: complex L x C column-major. */
WOFDM_API int wofdm_ber_run(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                  const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                  uint64_t seed, uint32_t variant,
                  int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot);
/* Same, but only frames f = shard_index (mod shard_count): one process per GPU sums the results
 * with a single all-reduce of the int64 counters (SURVEY.md section 8e).  (The channel-mask chain shards by contiguous
 * blocks of frames instead: wofdm_ber_run_masked_shard.) */
WOFDM_API int wofdm_ber_run_shard(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                        const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                        uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                        int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot);

/* Several window pairs on the SAME symbols in one call -- what the reference's loops do per frame: optimised and RC
 * windows on one signal_digmod with independent noise (python/ofdm_utils/wofdm_simulation.py:183-236), the RC window
 * and the six CaseA/CaseB steps of WOLA / CPW (matlab/main_BER_calculation.m:118-198).
 *   win_tx: n_var x n_tx doubles (pair v at win_tx + v*n_tx), win_rx: n_var x (N+tail_rx), n_var <= WOFDM_MAX_VARIANTS.
 *   bit_err / sym_err: n_var x n_snr (pair v at + v*n_snr); bit_tot / sym_tot: n_snr (the same for every pair).
 * Pair v gets exactly the counters of wofdm_ber_run_shard(..., variant + v, ...) with its windows: symbols depend on
 * (seed, frame), pair v's noise on (seed, frame, variant + v).  Where the tensor-core kernel applies, all pairs of a frame
 * are evaluated by ONE launch (symbols drawn once, tables of all pairs resident); otherwise one launch per pair. */
#define WOFDM_MAX_VARIANTS 8
WOFDM_API int wofdm_ber_run_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                        const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                        uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                        int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot);

/* The counters of wofdm_ber_run_multi resolved by sub-carrier and / or by channel realisation: where the errors come from
 * (guard-band edges, the bins a window protects, the deep-faded realisations that set the error floor).
 *   resolve: a non-empty combination of the flags below.  Cr = (resolve & WOFDM_BY_CHANNEL) ? C : 1,
 *            Nr = (resolve & WOFDM_BY_SUBCARRIER) ? N : 1 (FFT bin order, as wofdm_interf_power's sub-carrier axis).
 *   bit_err / sym_err: int64[n_var][n_snr][Cr][Nr]; sym_tot: int64[n_snr][Cr][Nr] (the same for every pair): this shard's
 *            frames of the cell times S-1 on active bins, 0 on guard bins; bit totals are sym_tot * bits.
 * Draws, noise numbering, window pairs (variant + v), sharding and the split over the handle's devices are those of
 * wofdm_ber_run_multi.  The call runs the resolved twin of the kernel wofdm_ber_run_multi picks for the same arguments (same
 * arithmetic): summed over the channel and bin axes, the counters equal that function's, bit for bit.  Where the twin's
 * per-sub-carrier accumulators do not fit the device's shared memory, the staged kernel runs instead with the same draws;
 * in fp32 its sums then agree up to decisions within rounding of a boundary (fp64 is staged on both sides: exact).  The
 * arrays are int64 and additive, so shards of several processes add up as the unresolved ones do.
 * WOFDM_EINVAL: resolve 0 or unknown bits, NULL buffers, a counter array whose size overflows, and what
 * wofdm_ber_run_multi rejects; WOFDM_ENOMEM: the device counter buffer cannot be allocated. */
#define WOFDM_BY_SUBCARRIER 1
#define WOFDM_BY_CHANNEL    2
WOFDM_API int wofdm_ber_run_resolved(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                       const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                       uint64_t seed, uint32_t variant, int shard_index, int shard_count, int resolve,
                       int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot);

/* Frame segments: a chosen subset of a job's frames.  The job has ensemble_max ensemble indices; its frames are numbered
 * as in wofdm_ber_run_multi with ensemble = ensemble_max, f = (snr_idx*C + c)*ensemble_max + e, and draw what they draw there.
 * Segment k = segments[3k .. 3k+2] = {snr_idx, e_begin, e_count} is every frame of that SNR point with any channel c < C
 * and e in [e_begin, e_begin + e_count).  A call runs its segments as one local index space j: segments in the order given,
 * channel-major, then e, inside a segment; shards and the handle's devices split j exactly as wofdm_ber_run_multi splits f
 * (device i of the handle takes j = shard_index + shard_count*i (mod shard_count*ndev)).  Every channel of a point gets
 * the same frames, so errors / total stays the reference's mean over channels of the mean over the ensemble, and the
 * counters of disjoint segment lists add up to those of their union: a finished run can be extended where it needs more
 * precision without repeating a frame.
 *   resolve = 0: bit_err / sym_err int64[n_var][n_snr], sym_tot int64[n_snr]; non-zero: the layout and semantics of
 *   wofdm_ber_run_resolved.  sym_tot counts this shard's frames; bit totals are sym_tot * bits.
 * The call runs the resolved-counter twins with the fallback rules of wofdm_ber_run_resolved.  The segment table is read
 * on the device, so the twin's counters of [0, e1) and [e1, E) add up to wofdm_ber_run_multi(E) / wofdm_ber_run_resolved(E).
 * WOFDM_EINVAL: n_seg < 1 or NULL segments; a segment outside [0, n_snr) x [0, ensemble_max) or with e_count < 1; two
 * overlapping segments of one point; ensemble_max < 1 or n_snr * C * ensemble_max overflowing int64; unknown resolve bits;
 * and what wofdm_ber_run_multi / _resolved reject.  The handle stays usable after every error. */
WOFDM_API int wofdm_ber_run_segments(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                       const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                       const int64_t* segments /* [n_seg][3] = {snr_idx, e_begin, e_count} */, int n_seg,
                       uint64_t seed, uint32_t variant, int shard_index, int shard_count, int resolve,
                       int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot);

/* Stopping rule of Monte-Carlo BER runs: every SNR point runs until it has counted `target` errors or ensemble_max ensemble
 * indices, in rounds of frame segments (wofdm_ber_run_segments; one plan for the whole call, one segment table upload,
 * one launch per device and one counter read per round).
 * Schedule (e_s: ensemble indices point s has run, b_s: its last block):
 *   round 0 gives every point b = min(first_block, ensemble_max);
 *   after each round, m_s = the minimum over the window pairs v of point s's cumulative bit errors (target_kind
 *   WOFDM_TARGET_BIT_ERRORS) or symbol errors (WOFDM_TARGET_SYMBOL_ERRORS);
 *   point s is done when m_s >= target or e_s == ensemble_max; otherwise its next block is
 *     min(ensemble_max - e_s, 2*b_s, m_s > 0 ? max(1, ceil((target - m_s) * e_s / m_s)) : 2*b_s)
 *   in exact integer arithmetic (128-bit, saturating);
 *   a round's segments are {s, e_s, b_s} of the active points in ascending SNR order.
 * reduce (optional): called once per round with this process's round counts int64[n_var][n_snr][2] = {bit, sym}, n =
 * 2*n_var*n_snr; it must overwrite them with their sum over the processes and return 0.  With it every process computes the
 * same schedule and returns the job's totals.  shard_count > 1 without reduce is WOFDM_EINVAL; a non-zero return fails the
 * call with WOFDM_EINVAL.  reduce must not call into this handle.
 * Outputs: ensemble_used[n_snr] (point s ran C * ensemble_used[s] frames: the ensemble indices [0, ensemble_used[s])),
 * bit_err / sym_err int64[n_var][n_snr] those frames' counters, bit_tot / sym_tot int64[n_snr] their totals, *rounds.
 * Bias: errors / bits of a run stopped at a target error count is not unbiased -- its relative bias is of order 1/target,
 * as in inverse binomial sampling; choose target >> 1 (100 gives ~1 %).  Points that stop at ensemble_max are unbiased.
 * WOFDM_EINVAL additionally: target < 1, an unknown target_kind, first_block < 1, NULL outputs. */
#define WOFDM_TARGET_BIT_ERRORS    0
#define WOFDM_TARGET_SYMBOL_ERRORS 1
typedef int (*wofdm_reduce_fn)(int64_t* counts, int64_t n, void* user);
WOFDM_API int wofdm_ber_run_adaptive(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx, int n_var,
                       const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max, int64_t first_block,
                       int target_kind, int64_t target, uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                       wofdm_reduce_fn reduce, void* reduce_user,
                       int64_t* ensemble_used, int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot, int* rounds);

/* Device-resident form: inputs are uploaded once, launches are asynchronous. */
WOFDM_API int wofdm_ber_plan_create(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                          const double* chan, int L, int C, const double* snr_db, int n_snr,
                          wofdm_ber_plan* plan);
/* The same for n_var window pairs (layout as in wofdm_ber_run_multi): counters are int64[n_var][n_snr][2] and
 * wofdm_ber_plan_read fills n_var x n_snr entries.  wofdm_ber_plan_variants returns n_var; *fused (optional) = 1 if one
 * launch evaluates all pairs. */
WOFDM_API int wofdm_ber_plan_create_multi(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                                int n_var, const double* chan, int L, int C, const double* snr_db, int n_snr,
                                wofdm_ber_plan* plan);
WOFDM_API int wofdm_ber_plan_variants(wofdm_ber_plan plan, int* fused);
/* Zeroes the plan's device counters and launches the shard on device slot `slot` of the handle,
 * on `stream` (a cudaStream_t; NULL = the plan's own stream).  Returns without synchronising.
 * One launch per slot and read: a second launch on the same slot before wofdm_ber_plan_read REPLACES the
 * first launch's counts (it waits for the first one if that ran on a different stream).
 * d_counters (optional out) = device pointer to int64[n_snr][2] = {bit_err, sym_err}. */
WOFDM_API int wofdm_ber_plan_launch(wofdm_ber_plan plan, int slot, int64_t ensemble, uint64_t seed, uint32_t variant,
                          int shard_index, int shard_count, void* stream, void** d_counters);
/* Waits for the launches and adds up the counters of the slots (devices) launched since the last read:
 * each slot contributes its most recent launch. */
WOFDM_API int wofdm_ber_plan_read(wofdm_ber_plan plan, int64_t* bit_err, int64_t* sym_err);
/* Name of the kernel variant the plan dispatches to (for logs / profiles). */
WOFDM_API const char* wofdm_ber_plan_kernel(wofdm_ber_plan plan);
WOFDM_API int wofdm_ber_plan_destroy(wofdm_ber_plan plan);

/* Verify mode: the caller injects every draw for F frames and gets the intermediates back.
 * Same chain and same kernels as wofdm_ber_run.
 *   chan: complex L x F (one channel per frame), snr_db: F, sym_idx: N x S x F constellation indices
 *   in the convention's own order, noise: complex len x F unit-variance draws with
 *   len = S*stride (noise_norm 0) or tail_tx + S*stride + L - 1 (noise_norm 1),
 *   eq_out: complex N x (S-1) x F, dec_idx: N x (S-1) x F, bit_err/sym_err: F.
 *   variant_kernel: 0 = the kernel wofdm_ber_run would pick, 1 = force the generic staged kernel,
 *   2 = the register-resident direct-form convolution over the whole frame (no tensor-core convolution, no
 *   circular interior), 3 = exclude the tensor-core convolution kernels only. */
WOFDM_API int wofdm_ber_verify(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                     const double* chan, int L, int F, const double* snr_db,
                     const int32_t* sym_idx, const double* noise, int variant_kernel,
                     double* eq_out, int32_t* dec_idx, int64_t* bit_err, int64_t* sym_err);
/* Exports the on-device draws of production frames frame_ids[0..F) so a production run can be
 * replayed through wofdm_ber_verify or a CPU oracle.  sym_idx: N x S x F, noise: complex len x F. */
WOFDM_API int wofdm_ber_draws(wofdm_handle h, const wofdm_sys_t* sys, int L, uint64_t seed, uint32_t variant,
                    const int64_t* frame_ids, int F, int32_t* sym_idx, double* noise);

/* ---- interference power ------------------------------------------------------------------ */
/* Replaces interf_power (python/ofdm_utils/interf_calc.py:20-113) per channel realisation:
 * P[k + N*c] = sum_{j!=k} |A_0[k,j]|^2 + sum_{m>=1} sum_j |A_m[k,j]|^2,  A_m = Rx_mat . H_m(h_c) . Tx_mat.
 * mode 0 = fp64 (DMMA), one contraction per channel and slice; 1 = TF32-split tensor cores (fp32 grade); 2 = fp64,
 * Hermitian form in the taps: A_m(c) = sum_l h_c[l] G_{m,l}, so the L impulse responses G go through the mode-0
 * contraction once per window pair and every channel costs L^2 MACs per sub-carrier (P_k = h^H Q_k h) -- the mode for
 * many channels (C > L; L <= 88).  chan: complex L x C, P: N x C column-major. */
WOFDM_API int wofdm_interf_power(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                       const double* chan, int L, int C, int mode, double* P);
/* MATLAB semantics (calculate_interference, matlab/main_interference_calculation.m:177-225):
 * scalar per channel, ISI slices summed before squaring.  P: C doubles. */
WOFDM_API int wofdm_interf_power_scalar(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx,
                              const double* win_rx, const double* chan, int L, int C, int mode, double* P);

/* Device times of the handle's last wofdm_interf_power* call, from CUDA events on its stream (ms; -1 = not taken:
 * kernel times exist for calls whose channels fit one batch): the whole call on the device (uploads, matrix builders,
 * band product, contraction, download), the band product B = H.Tx_mat alone, the tensor-core contraction alone.
 * k_slice0 / k_isi: rows of the real-form K dimension contracted for slice 0 / for every ISI slice (only the non-zero
 * prefix of an ISI slice exists), i.e. the executed GEMM is 2 * 2N * k * N flop per (channel, slice).  Any may be NULL. */
WOFDM_API int wofdm_interf_last_timing(wofdm_handle h, double* total_ms, double* band_ms, double* gemm_ms, int* k_slice0, int* k_isi);

/* ---- Channel-mask BER variant (next-row 8f-1) ----------------------------------------------------------------
 * run_sim_mc of matlab/main_channel_mask.m:334-360 for the MASKED signal: the guard-band frame (sys->guard = offset)
 * whose windowed symbols pass the DFT-domain raised-cosine mask of length 2 n_tx - 1 (dft_rc_filt, :398-417, roll_off
 * as `rollOff`, 10 in the reference); the filter tail of each symbol is added to the next one.  Same arguments, draws
 * (the symbol stream does not depend on `variant`) and counters as wofdm_ber_run, whose result with the same sys is
 * the UNMASKED ber of that script.  fp32, N = 128 / 256 / 512; the frames are split over the devices of the handle
 * (contiguous ranges of the global frame id: counters do not depend on the split).  The Tx side is one dense tensor-core
 * product (csrc/mask_gemm.cu: the script's matrices multiplied out once); WOFDM_MASK_FFT=1 in the environment selects
 * the per-symbol FFT kernel (csrc/mask_kernel.cuh) instead. */
WOFDM_API int wofdm_ber_run_masked(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                         uint64_t seed, uint32_t variant, int roll_off,
                         int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot);
/* wofdm_ber_run_masked for the frames of one shard: a CONTIGUOUS block of global frame ids
 * [floor(total*k/W), floor(total*(k+1)/W)), total = n_snr*C*ensemble, k = shard_index, W = shard_count -- not the
 * f = shard_index (mod shard_count) rule of wofdm_ber_run_shard: the mask product draws contiguous frame ranges, and the
 * handle's devices split this block as wofdm_ber_run_masked splits all frames.  *_tot count this shard's frames.  The
 * counters of the W shards add up to wofdm_ber_run_masked's, bit for bit, and wofdm_ber_run_masked is this call with
 * (0, 1).  Errors: those of wofdm_ber_run_masked, and WOFDM_EINVAL for a bad shard; the handle stays usable. */
WOFDM_API int wofdm_ber_run_masked_shard(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                         uint64_t seed, uint32_t variant, int roll_off, int shard_index, int shard_count,
                         int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot);
/* n_var window pairs of the channel-mask chain on the same frames in one call (1 <= n_var <= WOFDM_MAX_VARIANTS): pair v =
 * (win_tx + v*n_tx, win_rx + v*(N+tail_rx), roll_off[v]) gets exactly the counters of wofdm_ber_run_masked_shard with that
 * pair, variant + v and the same shard, bit for bit -- the symbols depend on (seed, frame) only, pair v's noise on (seed,
 * frame, variant + v).  Shards and the split over the handle's devices as in wofdm_ber_run_masked_shard.  A batch's symbols
 * are drawn once and one tensor-core product covers the mask matrices of all pairs; K1 evaluates all pairs of a frame in
 * one launch where its tables fit (else one launch per pair on the same product output).
 *   bit_err / sym_err: int64[n_var][n_snr]; bit_tot / sym_tot: int64[n_snr] (the same for every pair).
 * Errors: WOFDM_EINVAL for n_var outside [1, WOFDM_MAX_VARIANTS], a NULL roll_off, and what wofdm_ber_run_masked_shard
 * rejects for any pair (a roll-off that does not fit the mask among them).  The handle stays usable after every error. */
WOFDM_API int wofdm_ber_run_masked_multi(wofdm_handle h, const wofdm_sys_t* sys,
                         const double* win_tx /* n_var x n_tx */, const double* win_rx /* n_var x (N + tail_rx) */,
                         const int* roll_off /* n_var */, int n_var,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                         uint64_t seed, uint32_t variant, int shard_index, int shard_count,
                         int64_t* bit_err /* n_var x n_snr */, int64_t* bit_tot /* n_snr */,
                         int64_t* sym_err /* n_var x n_snr */, int64_t* sym_tot /* n_snr */);
/* The masked counters resolved as in wofdm_ber_run_resolved (resolve: a non-empty combination of WOFDM_BY_SUBCARRIER and
 * WOFDM_BY_CHANNEL; the same layout with n_var = 1): bit_err / sym_err int64[n_snr][Cr][Nr], sym_tot int64[n_snr][Cr][Nr]
 * = this shard's frames of the cell times S-1 on active bins, 0 on guard bins (bit totals: sym_tot * bits).  Shards as in
 * wofdm_ber_run_masked_shard.  Summed over the cells: wofdm_ber_run_masked_shard's counters, bit for bit -- the call runs
 * the resolved twin of the K1 kernel the masked chain picks (the same arithmetic and noise numbering).  Where a twin's
 * accumulators do not fit in shared memory, the staged twin runs with that kernel's noise numbering: it draws the same
 * noise, but its fp32 arithmetic differs, so the counters agree only up to decisions on a boundary.
 * Errors: WOFDM_EINVAL for a bad shard, a bad resolve, a NULL output or a counter array whose size overflows;
 * WOFDM_ENOMEM if the device counter buffer cannot be allocated; and what wofdm_ber_run_masked rejects.  The handle stays
 * usable after every error. */
WOFDM_API int wofdm_ber_run_masked_resolved(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble,
                         uint64_t seed, uint32_t variant, int roll_off, int shard_index, int shard_count, int resolve,
                         int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot);
/* Frame segments of the channel-mask chain: the segments, frame ids, draws and local index j of wofdm_ber_run_segments
 * (f = (snr_idx*C + c)*ensemble_max + e, the draws of wofdm_ber_run_masked(ensemble = ensemble_max); j runs over the
 * segments in the order given, channel-major, then e), so disjoint segment lists add up to the full masked run.  Shards
 * follow the masked chain's rule on j: shard k of W takes the contiguous block [floor(n_local*k/W), floor(n_local*(k+1)/W))
 * of the n_local local indices, and the handle's devices split that block contiguously.
 *   resolve = 0: bit_err / sym_err / sym_tot int64[n_snr]; non-zero: the [n_snr][Cr][Nr] layout of
 *   wofdm_ber_run_masked_resolved.  sym_tot counts this shard's frames; bit totals are sym_tot * bits.
 * The call always runs the resolved twin of the masked chain's K1 kernel, with the fallback rules of
 * wofdm_ber_run_masked_resolved.  Errors: what wofdm_ber_run_segments and wofdm_ber_run_masked_resolved reject (NULL or
 * empty, out-of-range or overlapping segments, e_count < 1, a bad shard, unknown resolve bits, NULL outputs, an overflowing
 * frame space or counter array, fp64, N outside {128, 256, 512}).  The handle stays usable after every error. */
WOFDM_API int wofdm_ber_run_masked_segments(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                         const int64_t* segments /* [n_seg][3] = {snr_idx, e_begin, e_count} */, int n_seg,
                         uint64_t seed, uint32_t variant, int roll_off, int shard_index, int shard_count, int resolve,
                         int64_t* bit_err, int64_t* sym_err, int64_t* sym_tot);
/* wofdm_ber_run_masked_segments for n_var window pairs on the same frames (1 <= n_var <= WOFDM_MAX_VARIANTS), as
 * wofdm_ber_run_masked_multi extends wofdm_ber_run_masked_shard: pair v = (win_tx + v*n_tx, win_rx + v*(N+tail_rx),
 * roll_off[v]) gets exactly what wofdm_ber_run_masked_segments gives with that pair and variant + v, bit for bit -- the
 * same segments, local indices, shard rule and device split.  A batch's symbols are drawn once and one tensor-core
 * product covers all pairs; the resolved twin of the K1 kernel evaluates all pairs of a frame in one launch where its
 * tables and accumulators fit, else one launch per pair on the same product output (the staged fallback of
 * wofdm_ber_run_masked_resolved keeps its fp32 caveat).  wofdm_ber_run_masked_segments is this call with n_var = 1.
 *   resolve = 0: bit_err / sym_err int64[n_var][n_snr], sym_tot int64[n_snr]; non-zero: bit_err / sym_err
 *   int64[n_var][n_snr][Cr][Nr], sym_tot int64[n_snr][Cr][Nr] (the same for every pair).
 * The resolved counters of several pairs over a whole job are this call with one segment {s, 0, ensemble} per point s.
 * Errors: WOFDM_EINVAL for n_var outside [1, WOFDM_MAX_VARIANTS], a NULL roll_off, and what
 * wofdm_ber_run_masked_segments rejects for any pair.  The handle stays usable after every error. */
WOFDM_API int wofdm_ber_run_masked_segments_multi(wofdm_handle h, const wofdm_sys_t* sys,
                         const double* win_tx /* n_var x n_tx */, const double* win_rx /* n_var x (N + tail_rx) */,
                         const int* roll_off /* n_var */, int n_var,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                         const int64_t* segments /* [n_seg][3] = {snr_idx, e_begin, e_count} */, int n_seg,
                         uint64_t seed, uint32_t variant, int shard_index, int shard_count, int resolve,
                         int64_t* bit_err /* [n_var][n_snr] or [n_var][n_snr][Cr][Nr] */, int64_t* sym_err,
                         int64_t* sym_tot /* [n_snr] or [n_snr][Cr][Nr] */);
/* run_sim_mc of matlab/main_channel_mask.m with the stopping rule of wofdm_ber_run_adaptive: the masked and the unmasked
 * chain on the same frames (one window pair, the same sys), every SNR point run until both have counted `target` errors
 * or ensemble_max ensemble indices.
 *   row 0 of bit_err / sym_err (int64[2][n_snr]): the masked chain (wofdm_ber_run_masked_segments), noise stream
 *   variant + 1; row 1: the unmasked chain (wofdm_ber_run_segments), noise stream variant.  variant = 0 gives the draws
 *   of the two calls run_sim_mc makes.
 * The schedule is wofdm_ber_run_adaptive's with m_s the minimum over the two rows.  Each row shards by its own chain's
 * rule (contiguous blocks of the round's local indices for row 0, j = shard_index (mod shard_count) for row 1); reduce
 * receives this process's round counts int64[2][n_snr][2] = {bit, sym} (n = 4*n_snr) and makes them the job's.
 * shard_count > 1 without reduce is WOFDM_EINVAL.  Outputs: ensemble_used[n_snr], bit_tot / sym_tot int64[n_snr] (the
 * same for both rows), *rounds.  The stopped estimator has the relative bias of order 1/target that wofdm_ber_run_adaptive
 * states; points that stop at ensemble_max are unbiased.  Errors: those of wofdm_ber_run_adaptive and of
 * wofdm_ber_run_masked; the handle stays usable. */
WOFDM_API int wofdm_ber_run_masked_adaptive(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, const double* win_rx,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max, int64_t first_block,
                         int target_kind, int64_t target, uint64_t seed, uint32_t variant, int roll_off, int shard_index,
                         int shard_count, wofdm_reduce_fn reduce, void* reduce_user,
                         int64_t* ensemble_used, int64_t* bit_err, int64_t* bit_tot, int64_t* sym_err, int64_t* sym_tot, int* rounds);
/* wofdm_ber_run_masked_adaptive for n_var window pairs / roll-offs on the same frames (1 <= n_var <= WOFDM_MAX_VARIANTS),
 * pair v = (win_tx + v*n_tx, win_rx + v*(N+tail_rx), roll_off[v]).  2 n_var rows of counters, bit_err / sym_err
 * int64[2][n_var][n_snr]:
 *   block 0, row v: the masked chain of pair v (wofdm_ber_run_masked_segments_multi), noise stream variant + n_var + v;
 *   block 1, row v: the unmasked chain of pair v (wofdm_ber_run_segments with n_var pairs), noise stream variant + v.
 * These are the streams of ofdm_utils.run_sim_mc_multi; with n_var = 1 (masked variant + 1, unmasked variant) those of
 * wofdm_ber_run_masked_adaptive, which is this call with n_var = 1.  The schedule is wofdm_ber_run_adaptive's over the
 * 2 n_var rows: a point stops when every row has counted `target` errors, or at ensemble_max.  Sharding as in
 * wofdm_ber_run_masked_adaptive; reduce receives int64[2][n_var][n_snr][2] = {bit, sym} (n = 4*n_var*n_snr).  Outputs:
 * ensemble_used[n_snr], bit_tot / sym_tot int64[n_snr] (the same for every row), *rounds.  Errors: WOFDM_EINVAL for n_var
 * outside [1, WOFDM_MAX_VARIANTS], a NULL roll_off, and what wofdm_ber_run_masked_adaptive rejects for any pair; the
 * handle stays usable. */
WOFDM_API int wofdm_ber_run_masked_adaptive_multi(wofdm_handle h, const wofdm_sys_t* sys,
                         const double* win_tx /* n_var x n_tx */, const double* win_rx /* n_var x (N + tail_rx) */,
                         const int* roll_off /* n_var */, int n_var,
                         const double* chan, int L, int C, const double* snr_db, int n_snr, int64_t ensemble_max,
                         int64_t first_block, int target_kind, int64_t target, uint64_t seed, uint32_t variant,
                         int shard_index, int shard_count, wofdm_reduce_fn reduce, void* reduce_user,
                         int64_t* ensemble_used, int64_t* bit_err /* [2][n_var][n_snr] */, int64_t* bit_tot,
                         int64_t* sym_err /* [2][n_var][n_snr] */, int64_t* sym_tot, int* rounds);

/* ---- Window-optimisation Hessian (next-row 8f-2) -------------------------------------------------------------
 * The quadratic form of the interference power in the reduced window variables: OptimizerTx / OptimizerRx /
 * OptimizerTxRx.gen_hessian (python/optimization_tools/optimizers.py:232-257, 387-410, 808-833) and
 * quad_objective_tx / _rx (matlab/window_optimization.m:596-680), whose O(n^2 N^2) loops are the slowest part of the
 * reference's run_opt.  chan: ONE impulse response, complex L (the reference passes the mean of the stored set).
 * H: n_var x n_var doubles (symmetric), n_var = (tail_rx/2 + 1) * (tail_tx + 1), variable index
 * u = a*(tail_tx+1) + b for Rx-tail variable a and Tx-tail variable b (OptimizerTxRx's flatten order; Tx-only and
 * Rx-only systems have tail_rx = 0 or tail_tx = 0 and the index is b or a).  *n_var (may be NULL) returns n_var. */
WOFDM_API int wofdm_window_hessian(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, double* H, int* n_var);
/* The two parts of that quadratic form for ARBITRARY basis windows: basis_tx = n_tb windows of n_tx samples, basis_rx = n_rb
 * windows of N + tail_rx samples (row-major), variable u = a*n_tb + b, n_var = n_rb*n_tb:
 *   H_ici[u,u'] = 2 Re <offdiag A0_u, offdiag A0_u'>,   H_isi[u,u'] = 2 Re <AS_u, AS_u'>   (wofdm_window_hessian = their sum
 * on the reduced bases).  With the FULL window as the variable (basis = identity) and the other side's window fixed (one
 * row) these are quad_objective_tx / _rx of matlab/window_optimization.m:596-680:
 *   HTx (or HRx) = alpha * H_ici + (1 - alpha) * diag(row sums of H_isi)       (H2 = real(diag(diag(B2' B2 C C'))), :628-631). */
WOFDM_API int wofdm_window_hessian_parts(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L,
                               const double* basis_tx, int n_tb, const double* basis_rx, int n_rb, double* H_ici, double* H_isi);
/* Mean over a channel set of wofdm_window_hessian: H = (1/C) sum_c H(h_c), the quadratic form of the EXPECTED interference
 * power over the set (the reference optimises against the mean impulse response, one random channel of covariance R/C).
 * chan: complex L x C column-major (channels/vehicularA.npy layout).  Same variable order, same n_var.
 * H(h) is a linear function of h h^H, so the mean equals sum_j H(g_j) for any factor sum_j g_j g_j^H of the sample tap
 * covariance R = (1/C) sum_c h_c h_c^H.  C <= L: the channels themselves (C passes, weight 1/C; C = 1 gives exactly
 * wofdm_window_hessian).  C > L: R is formed in fp64 on the host and factored by a pivoted Cholesky decomposition into
 * r = rank(R) <= L virtual channels; directions whose remaining variance is at most 1e-14 of the largest diagonal entry of
 * R are dropped.  One pass of the device pipeline per virtual channel, the Gram products summed on the device, one download.
 * Runs on device slot 0 of the handle only (a multi-device handle gives the single-device result).
 * WOFDM_EINVAL: C < 1, NULL buffers, non-finite taps, or what wofdm_window_hessian rejects; N % 64 != 0: WOFDM_EUNSUPPORTED. */
WOFDM_API int wofdm_window_hessian_set(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, int C, double* H, int* n_var);
/* Mean over the set of the two parts of wofdm_window_hessian_parts (arbitrary bases, MATLAB quad_objective semantics): same
 * factor and passes as wofdm_window_hessian_set, H_ici and H_isi each the mean of the per-channel parts. */
WOFDM_API int wofdm_window_hessian_parts_set(wofdm_handle h, const wofdm_sys_t* sys, const double* chan, int L, int C,
                                             const double* basis_tx, int n_tb, const double* basis_rx, int n_rb, double* H_ici, double* H_isi);
/* Of the handle's last wofdm_window_hessian* call: device time from the first upload to the end of the download (CUDA events
 * on its stream, ms; -1 = not taken), host time of the channel-set factorisation (ms; 0 for a single channel) and the passes
 * of the device pipeline (virtual channels).  Any may be NULL. */
WOFDM_API int wofdm_window_hessian_last_timing(wofdm_handle h, double* device_ms, double* factor_ms, int* passes);

/* ---- Channel generation (next-row 8f-4) ------------------------------------------------------------------
 * ITU-R tapped-delay-line channels with GMEDS_1 Rayleigh fading on the device: channel_model.gen_chan
 * (python/channel_model/itur_channels.py:33-94 + rayleigh_fading.py:52-102), the producer of channels/<standard>.npy
 * (python/wofdm_optimization.py:63-86).
 *   wofdm_channel_profile: "vehicularA" | "vehicularB" | "outdoor-indoorA" | "outdoor-indoorB" -> index, or WOFDM_EINVAL.
 *   One SET = one call of the reference's gen_chan: its own oscillator phases, no_frames time samples frame_duration
 *   apart, every path scaled to ENERGY 10^(dB/10) over the set (the reference's adjust_power).  The reference's
 *   driver stores C channels as C sets of one frame each: n_sets = C, no_frames = 1.
 *   phases: NULL -> Philox4x32-10 + Box-Muller draws keyed by (seed, set); else the standard-normal draws themselves,
 *   [n_sets][n_paths][21][2] in the reference's draw order (path, oscillator, real part / imaginary part).
 *   chan: complex L x (n_sets*no_frames) column-major, column = set*no_frames + frame. */
WOFDM_API int wofdm_channel_profile(const char* standard);
WOFDM_API int wofdm_gen_channels(wofdm_handle h, int profile, int L, double doppler_freq, double sampling_rate,
                       double frame_duration, int no_frames, int n_sets, uint64_t seed, const double* phases,
                       double* chan);

/* Next row 8f-3: PSD / out-of-band-radiation estimate of the windowed Tx signal.  Replaces the signal construction of
 * wOFDMSystem.estimate_obr and __psd_estimate (python/ofdm_utils/timefreq_simulation.py:104-123, 216-253; MATLAB twin
 * matlab/main_OOB_figures.m:121-159): records of n_sym OFDM symbols on the sub-carrier allocation of :223-232 (DC and the
 * 2*guard_band - 1 centre bins null, N - 2*guard_band data rows), IDFT, CP/CS, Tx window win_tx (N + cp + cs values),
 * overlap-add of the tails (tail_tx = 0: plain serialisation, as the reference does for the un-windowed signals), cut
 * into slices of 8N samples (the last, partial one zero padded), |fftshift(FFT)|^2 averaged over slices and records.
 *   sym_idx: int32 [records][n_sym][N - 2*guard_band] injected constellation indices (records = 1 reproduces the
 *   reference's estimator for its draw), or NULL: on-device Philox draws keyed by (seed, record, symbol).
 *   psd: 8N doubles, the reference's X_est (fftshifted).  N = 256. */
WOFDM_API int wofdm_psd_estimate(wofdm_handle h, int N, int cp, int cs, int tail_tx, int bits, int constellation,
                       const double* win_tx, int guard_band, int n_sym, int64_t records, uint64_t seed,
                       const int32_t* sym_idx, double* psd);

/* PSD of the channel-mask chain's Tx streams (matlab/main_channel_mask.m), masked and unmasked, on the frames of its BER
 * calls: frames f0 .. f0 + n_frames - 1 carry exactly the symbols wofdm_ber_run_masked / wofdm_ber_run give frame f with
 * the same seed (wofdm_ber_draws exports them).  A frame is sys->S symbols on the guard-band allocation (sys->guard),
 * windowed with win_tx (n_tx values), overlap-added with the frame stride into tail_tx + S * stride samples; the masked
 * stream passes the mask of roll_off bins exactly as in the BER chain (the last symbol's filter tail is dropped), the
 * unmasked one is the same symbols without it.  Each non-NULL output gets the 8N-point fftshifted PSD averaged over
 * the slices of every frame; a NULL output skips that half of the work, and at least one must be non-NULL.  Ranges add
 * up: the PSD of [a, c) is the frame-weighted mean of [a, b) and [b, c) up to the order of fp64 additions.
 *   estimator 0: __psd_estimate of the reference (python/ofdm_utils/timefreq_simulation.py:104-123, as
 *                wofdm_psd_estimate): floor(len / 8N) non-overlapping slices plus the zero-padded remainder, averaged over
 *                floor + 1 slices.
 *   estimator 1: Hann-tapered slices w[n] = sin^2(pi n / 8N) at a hop of 4N (50 % overlap), no remainder slice, each
 *                periodogram scaled by 8N / sum(w^2) = 8/3 (a white stream reads the same level under both).
 * The Tx fields of sys as wofdm_ber_run_masked accepts them (fp32, N = 128 / 256 / 512, bits < 8 with a guard band,
 * roll_off that fits the mask); the Rx fields are ignored.  Device slot 0 only.  Errors: WOFDM_EINVAL for a NULL win_tx,
 * both outputs NULL, f0 < 0, n_frames < 1, an overflowing frame range, a bad estimator or roll_off, or a stream shorter
 * than one slice (tail_tx + S * stride < 8N); WOFDM_EUNSUPPORTED for fp64, another N, or a frame the mask product's
 * symbol kernel cannot hold in shared memory.  The handle stays usable after every error. */
WOFDM_API int wofdm_psd_masked(wofdm_handle h, const wofdm_sys_t* sys, const double* win_tx, int roll_off,
                       uint64_t seed, int64_t f0, int64_t n_frames, int estimator,
                       double* psd_masked /* 8N or NULL */, double* psd_unmasked /* 8N or NULL */);
/* wofdm_psd_masked for n_var Tx windows / roll-offs on the same frames (1 <= n_var <= WOFDM_MAX_VARIANTS): spectrum v of
 * psd_masked / psd_unmasked (row v of n_var x 8N) is wofdm_psd_masked's with win_tx + v*n_tx and roll_off[v], up to the
 * order of fp64 additions.  Every requested spectrum is one pair of a single mask product (the unmasked ones with a unit
 * impulse for the mask): a batch's symbols are drawn once, and one product and one PSD launch cover all spectra.  A NULL
 * output skips that half for every configuration.  wofdm_psd_masked is this call with n_var = 1.  Errors: WOFDM_EINVAL
 * for n_var outside [1, WOFDM_MAX_VARIANTS], a NULL roll_off, and what wofdm_psd_masked rejects for any roll_off[v]; the
 * handle stays usable. */
WOFDM_API int wofdm_psd_masked_multi(wofdm_handle h, const wofdm_sys_t* sys,
                       const double* win_tx /* n_var x n_tx */, const int* roll_off /* n_var */, int n_var,
                       uint64_t seed, int64_t f0, int64_t n_frames, int estimator,
                       double* psd_masked /* n_var x 8N or NULL */, double* psd_unmasked /* n_var x 8N or NULL */);

#ifdef __cplusplus
}
#endif
#endif /* WOFDM_H_ */
