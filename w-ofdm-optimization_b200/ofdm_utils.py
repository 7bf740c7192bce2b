"""Host-side mirror of the reference's hot-path interface, backed by libwofdm.so.

Same names, argument meaning, file side effects and error behaviour (Python exceptions) as

* ``ofdm_utils.simulation_fun(data)``            python/ofdm_utils/wofdm_simulation.py:20-73
* ``wOFDMSystem(...).run_simulation(...)``       python/ofdm_utils/wofdm_simulation.py:368-481
* ``ofdm_utils.interf_power(sys, [Vtx, Vrx], N, cp, tail_tx, tail_rx)``   python/ofdm_utils/interf_calc.py:20-113
* ``run_simulation(ensemble, symbolsPerTx, ...)`` matlab/main_BER_calculation.m:230-274 (what the MEX gateway calls)
* ``calculate_interference(cpLength, typeOFDM, windowTx, windowRx, ...)`` matlab/main_interference_calculation.m:177-225
* ``run_sim_mc(...)`` / ``psd_sim_mc(...)``         matlab/main_channel_mask.m: the masked chain's BER and Tx spectra

so a reference driver switches backend by importing this module instead of ``ofdm_utils`` (INTEGRATION.md).
Everything numeric happens on the GPU through the C-ABI; there is no CPU fallback.  Documented deviations:
the Monte-Carlo draws come from the on-device Philox streams (not numpy's / MATLAB's global generators), and
the MATLAB BER is averaged over the whole ensemble (the reference overwrites it each iteration, SURVEY F6).
"""
from __future__ import annotations

import os

import numpy as np

from . import capi

_HANDLE = None
TX_SYSTEMS = ("CPW", "WOLA", "CPwtx", "wtx")
RX_SYSTEMS = ("CPW", "WOLA", "CPwrx", "wrx")


def default_handle():
    """Process-wide handle on the current device(s) (LOCAL_RANK under torchrun, else every visible GPU)."""
    global _HANDLE
    if _HANDLE is None:
        lr = os.environ.get("LOCAL_RANK")
        _HANDLE = capi.Handle([int(lr)] if lr is not None else None)
    return _HANDLE


def set_handle(h):
    global _HANDLE
    _HANDLE = h


def _diag(w):
    """Windows cross the reference boundary as dense diagonal matrices (SURVEY section 8b)."""
    w = np.asarray(w, dtype=np.float64)
    return np.diag(w).copy() if w.ndim == 2 else w.ravel()


class wOFDMSystem:
    """Mirror of the reference class: parameter table + run_simulation writing the SER .npy files."""

    def __init__(self, system_design: str, dft_len: int, cp_len: int, tail_tx: int, tail_rx: int, folder_path: str,
                 seed: int = 0, precision: int = 0, handle=None):
        self.name = system_design
        self.dft_len, self.cp_len, self.tail_tx, self.tail_rx = dft_len, cp_len, tail_tx, tail_rx
        self.folder_path = folder_path
        self.seed, self.precision = seed, precision
        self._h = handle
        s = capi.params_from_name(system_design, dft_len, cp_len, tail_tx, tail_rx)   # raises on unknown names
        self.cs_len, self.rm_len, self.shift_len = s.cs, s.rm, s.shift

    def _sys(self, no_symbols, bits=4):
        return capi.params_from_name(self.name, self.dft_len, self.cp_len, self.tail_tx, self.tail_rx, bits=bits,
                                     S=no_symbols, noise_norm=0, constellation=0, precision=self.precision)

    def run_simulation(self, channel_models, window_tx, window_rx, ensemble, snr_arr, no_symbols):
        """SER of the optimised and the RC windows on the same symbols with independent noise
        (wofdm_simulation.py:183-236), saved as ser/opt_<sys>_<cp>.npy, ser/rc_<sys>_<cp>.npy (CP: ser/CP_<cp>.npy)."""
        h = self._h or default_handle()
        path_to_ser = os.path.join(self.folder_path, "ser")
        os.makedirs(path_to_ser, exist_ok=True)
        s = self._sys(int(no_symbols))
        snr = np.asarray(snr_arr, dtype=np.float64)
        if self.name == "CP":
            r = h.ber_run(s, np.ones(s.n_tx), np.ones(s.N + s.tail_rx), channel_models, snr, ensemble, seed=self.seed)
            ser = r["sym_err"] / r["sym_tot"]
            np.save(os.path.join(path_to_ser, f"CP_{self.cp_len}.npy"), ser)
            return ser
        # ONE call (one launch where the tensor-core kernel applies): both window pairs on every frame's symbols
        r = h.ber_run_multi(s, [_diag(window_tx), capi.rc_window_tx(s)], [_diag(window_rx), capi.rc_window_rx(s)],
                            channel_models, snr, ensemble, seed=self.seed, variant=0)
        ser_opt, ser_rc = r["sym_err"][0] / r["sym_tot"], r["sym_err"][1] / r["sym_tot"]
        np.save(os.path.join(path_to_ser, f"opt_{self.name}_{self.cp_len}.npy"), ser_opt)
        np.save(os.path.join(path_to_ser, f"rc_{self.name}_{self.cp_len}.npy"), ser_rc)
        return ser_opt, ser_rc

    def run_simulation_per_subcarrier(self, channel_models, window_tx, window_rx, ensemble, snr_arr, no_symbols):
        """run_simulation resolved by sub-carrier: the same symbols and noise (same seed), SER of shape (n_snr, N) per
        FFT bin for the optimised and the RC windows ((ser_opt, ser_rc); 'CP': one array).  Writes no files.  The
        mean over the active bins is run_simulation's SER."""
        h = self._h or default_handle()
        s = self._sys(int(no_symbols))
        snr = np.asarray(snr_arr, dtype=np.float64)
        if self.name == "CP":
            wt, wr = [np.ones(s.n_tx)], [np.ones(s.N + s.tail_rx)]
        else:
            wt, wr = [_diag(window_tx), capi.rc_window_tx(s)], [_diag(window_rx), capi.rc_window_rx(s)]
        r = h.ber_run_resolved(s, wt, wr, channel_models, snr, ensemble, seed=self.seed, variant=0, by_subcarrier=True)
        tot = r["sym_tot"][:, 0, :]
        ser = [np.divide(e[:, 0, :], tot, out=np.zeros(tot.shape), where=tot > 0) for e in r["sym_err"]]
        return ser[0] if self.name == "CP" else (ser[0], ser[1])

    def run_simulation_adaptive(self, channel_models, window_tx, window_rx, ensemble_max, snr_arr, no_symbols,
                                target_errors, first_block=1):
        """run_simulation with a stopping rule: each SNR point runs until both window pairs have counted target_errors
        symbol errors (the python convention counts symbols) or ensemble_max ensemble indices (Handle.ber_run_adaptive).
        Frame f of a point is the frame run_simulation(ensemble=ensemble_max) draws.  Returns (ser_opt, ser_rc,
        ensemble_used) ('CP': (ser, ensemble_used)); writes no files."""
        h = self._h or default_handle()
        s = self._sys(int(no_symbols))
        snr = np.asarray(snr_arr, dtype=np.float64)
        if self.name == "CP":
            wt, wr = [np.ones(s.n_tx)], [np.ones(s.N + s.tail_rx)]
        else:
            wt, wr = [_diag(window_tx), capi.rc_window_tx(s)], [_diag(window_rx), capi.rc_window_rx(s)]
        r = h.ber_run_adaptive(s, wt, wr, channel_models, snr, ensemble_max, target_symbol_errors=int(target_errors),
                               first_block=first_block, seed=self.seed, variant=0)
        ser = [e / r["sym_tot"] for e in r["sym_err"]]
        return (ser[0], r["ensemble_used"]) if self.name == "CP" else (ser[0], ser[1], r["ensemble_used"])


def load_window_tails(system_design, window_path, cp_len, tail_tx, tail_rx):
    """<window_path>/<sys>_<cp>.npy -> (x_tx, x_rx) reduced variables (wofdm_simulation.py:46-66, SURVEY App. A.4)."""
    if system_design == "CP":
        return np.array([1.0]), np.array([1.0])
    x = np.load(os.path.join(window_path, f"{system_design}_{cp_len}.npy")).ravel()
    if system_design in ("WOLA", "CPW"):
        return x[:tail_tx + 1], x[tail_tx + 1:]
    if system_design in ("wtx", "CPwtx"):
        return x, np.array([1.0])
    if system_design in ("wrx", "CPwrx"):
        return np.array([1.0]), x
    raise ValueError(f"unknown w-OFDM system {system_design!r}")


def simulation_fun(data: tuple, seed: int = 0, handle=None):
    """Drop-in for ofdm_utils.simulation_fun: same 11-tuple
    (system_design, dft_len, cp_len, tail_tx, tail_rx, channel_path, window_path, ensemble, snr_arr, no_symbols,
    folder_path), same input files, same output files."""
    system_design, dft_len, cp_len, tail_tx, tail_rx = data[0:5]
    channel_path, window_path, ensemble, snr_arr, no_symbols, folder_path = data[5:]
    channel_models = np.load(channel_path)
    x_tx, x_rx = load_window_tails(system_design, window_path, cp_len, tail_tx, tail_rx)
    s = capi.params_from_name(system_design, dft_len, cp_len, tail_tx, tail_rx)
    win_tx = capi.expand_window_tx(s, x_tx)          # reduce_variable_tx @ tail   (wofdm_simulation.py:67-68)
    win_rx = capi.expand_window_rx(s, x_rx)          # reduce_variable_rx @ tail   (:69)
    model = wOFDMSystem(system_design, dft_len, cp_len, tail_tx, tail_rx, folder_path, seed=seed, handle=handle)
    return model.run_simulation(channel_models, win_tx, win_rx, ensemble, snr_arr, no_symbols)


def interf_power(sys_design: str, window_data: list, dft_len: int, cp_len: int, tail_tx: int, tail_rx: int,
                 channel_path: str = "channels/vehicularA.npy", per_channel: bool = False, mode=None, handle=None):
    """Drop-in for ofdm_utils.interf_power.  Default: the reference's behaviour -- the MEAN impulse response of the
    stored set (interf_calc.py:80-83) -> (P_opt, P_rc), each (N,), or a single (N,) vector for 'CP'.
    per_channel=True evaluates every realisation: arrays of shape (C, N).  mode None: fp64, the direct contraction
    (0) for up to L channels, the Hermitian form in the taps (2) for more."""
    h = handle or default_handle()
    chann = np.load(channel_path)
    chan = chann if per_channel else chann.mean(axis=1)[:, None]
    if mode is None:
        mode = 2 if (chan.shape[1] > chan.shape[0] and chan.shape[0] <= 88) else 0
    if sys_design == "CP":                                             # interf_calc.py:57-73
        s = capi.params_from_name("CP", dft_len, cp_len, 0, 0)
        P = h.interf_power(s, np.ones(s.n_tx), np.ones(s.N), chan, mode=mode)
        return P if per_channel else P[0]
    s = capi.params_from_name(sys_design, dft_len, cp_len, tail_tx, tail_rx)
    v_tx, v_rx = window_data
    P_opt = h.interf_power(s, _diag(v_tx), _diag(v_rx), chan, mode=mode)
    P_rc = h.interf_power(s, capi.rc_window_tx(s), capi.rc_window_rx(s), chan, mode=mode)
    return (P_opt, P_rc) if per_channel else (P_opt[0], P_rc[0])


# ---- MATLAB-side signatures (what mex/wofdm_mex.cpp marshals) -----------------------------------------

def run_simulation(ensemble, symbolsPerTx, bitsPerSubcarrier, numSubcar, cpLength, csLength, windowTx, channel, snr,
                   tailTx, tailRx, windowRx, prefixRemovalLength, circularShiftLength, seed=0, handle=None):
    """BER of one (window pair, channel, SNR) -- positional arguments of matlab/main_BER_calculation.m:230-232.
    Gray unit-power QAM, bit errors over numSubcar*bits*(symbolsPerTx-1) bits per frame, noise normalised on
    the full convolution (:260).  Returns errors/bits over the WHOLE ensemble."""
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcarrier),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0)
    r = h.ber_run(s, _diag(windowTx), _diag(windowRx), np.asarray(channel).ravel(), [float(snr)], int(ensemble), seed=seed)
    return float(r["bit_err"][0] / r["bit_tot"][0])


def run_simulation_multi(ensemble, symbolsPerTx, bitsPerSubcarrier, numSubcar, cpLength, csLength, windowsTx, channel, snr,
                         tailTx, tailRx, windowsRx, prefixRemovalLength, circularShiftLength, seed=0, handle=None):
    """The window variants main_BER_calculation.m evaluates per (channel, SNR) -- {optimised, RC} for wtx / wrx (:66-117),
    RC + CaseA steps 1-3 + CaseB steps 1-3 for WOLA / CPW (:118-198) -- in ONE call on the same bits: windowsTx / windowsRx
    are lists of n_var diagonal matrices (or vectors); returns n_var BERs, variant v with the noise stream of
    run_simulation(..., seed) called with variant v."""
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcarrier),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0)
    r = h.ber_run_multi(s, [_diag(w) for w in windowsTx], [_diag(w) for w in windowsRx], np.asarray(channel).ravel(),
                        [float(snr)], int(ensemble), seed=seed)
    return r["bit_err"][:, 0] / r["bit_tot"][0]


def run_sim_mc(ensemble, cpLength, csLength, tailTx, tailRx, windowTx, windowRx, channel, snr, offset,
               prefixRemovalLength, circularShiftLength, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff, seed=0, handle=None):
    """[berMasked, ber] of one (window pair, channel, SNR) -- positional arguments of run_sim_mc,
    matlab/main_channel_mask.m:334-337: numSubcar - 2*offset active sub-carriers, the same symbols with and without the
    DFT-domain raised-cosine mask, independent noise.  Errors / bits over the whole ensemble."""
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    wt, wr, ch = _diag(windowTx), _diag(windowRx), np.asarray(channel).ravel()
    r = h.ber_run(s, wt, wr, ch, [float(snr)], int(ensemble), seed=seed, variant=0)
    rm = h.ber_run_masked(s, wt, wr, ch, [float(snr)], int(ensemble), seed=seed, variant=1, roll_off=int(rollOff))
    return float(rm["bit_err"][0] / rm["bit_tot"][0]), float(r["bit_err"][0] / r["bit_tot"][0])


def run_sim_mc_multi(ensemble, cpLength, csLength, tailTx, tailRx, windowTx, windowRx, channel, snr, offset,
                     prefixRemovalLength, circularShiftLength, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff, seed=0,
                     handle=None):
    """run_sim_mc for n_var configurations on the same symbols in one masked and one unmasked call: windowTx, windowRx and
    rollOff are lists of n_var (diagonal matrices or vectors; integers).  Returns (berMasked, ber), arrays of n_var.
    Configuration v's unmasked chain has noise stream v (Handle.ber_run_multi), its masked chain n_var + v
    (Handle.ber_run_masked_multi), so no two streams meet; with one configuration this is run_sim_mc's result exactly."""
    wts, wrs, ros = list(windowTx), list(windowRx), list(np.atleast_1d(rollOff))
    if not (len(wts) == len(wrs) == len(ros)) or not wts:
        raise ValueError(f"windowTx, windowRx and rollOff must be lists of the same length "
                         f"(got {len(wts)}, {len(wrs)}, {len(ros)})")
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    wt, wr, ch = [_diag(w) for w in wts], [_diag(w) for w in wrs], np.asarray(channel).ravel()
    nv = len(wt)
    r = h.ber_run_multi(s, wt, wr, ch, [float(snr)], int(ensemble), seed=seed, variant=0)
    rm = h.ber_run_masked_multi(s, wt, wr, ch, [float(snr)], int(ensemble), seed=seed, variant=nv,
                                roll_offs=[int(x) for x in ros])
    return rm["bit_err"][:, 0] / rm["bit_tot"][0], r["bit_err"][:, 0] / r["bit_tot"][0]


def run_sim_mc_per_subcarrier(ensemble, cpLength, csLength, tailTx, tailRx, windowTx, windowRx, channel, snr, offset,
                              prefixRemovalLength, circularShiftLength, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff, seed=0,
                              handle=None):
    """run_sim_mc resolved by sub-carrier: (berMasked, ber), each of shape (numSubcar,) in FFT bin order, 0 on the guard
    bins -- where the mask costs errors.  The same symbols with and without the mask, the noise of run_sim_mc with the
    same seed, so the mean over the active bins is run_sim_mc's result."""
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    wt, wr, ch = _diag(windowTx), _diag(windowRx), np.asarray(channel).ravel()
    r = h.ber_run_resolved(s, [wt], [wr], ch, [float(snr)], int(ensemble), seed=seed, variant=0, by_subcarrier=True)
    rm = h.ber_run_masked_resolved(s, wt, wr, ch, [float(snr)], int(ensemble), seed=seed, variant=1, roll_off=int(rollOff),
                                   by_subcarrier=True)
    out = []
    for be, bt in ((rm["bit_err"][0, 0], rm["bit_tot"][0, 0]), (r["bit_err"][0, 0, 0], r["bit_tot"][0, 0])):
        out.append(np.divide(be, bt, out=np.zeros(bt.shape), where=bt > 0))
    return out[0], out[1]


def run_sim_mc_adaptive(ensemble_max, cpLength, csLength, tailTx, tailRx, windowTx, windowRx, channel, snr, offset,
                        prefixRemovalLength, circularShiftLength, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff,
                        target_bit_errors, first_block=1, seed=0, handle=None):
    """run_sim_mc with each SNR point stopped at a bit-error target (wofdm_ber_run_masked_adaptive): every point runs until
    both the masked and the unmasked chain have counted target_bit_errors bit errors, or ensemble_max ensemble indices.
    channel: one impulse response, or C x L (rows = realisations); snr: a scalar or a vector.  Returns (berMasked, ber,
    ensemble_used), arrays over the SNR points, and writes no files.  An unreachable target gives run_sim_mc's result for
    ensemble = ensemble_max."""
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    ch = np.atleast_2d(np.asarray(channel)).T                         # (L, C)
    r = h.ber_run_masked_adaptive(s, _diag(windowTx), _diag(windowRx), ch, np.atleast_1d(np.asarray(snr, dtype=np.float64)),
                                  int(ensemble_max), target_bit_errors=int(target_bit_errors), first_block=int(first_block),
                                  seed=seed, variant=0, roll_off=int(rollOff))
    return r["bit_err"][0] / r["bit_tot"], r["bit_err"][1] / r["bit_tot"], r["ensemble_used"]


def _roll_off_list(rollOff, n_var):
    """rollOff as n_var integers: one value for every configuration, or a list of n_var"""
    ros = [int(x) for x in np.atleast_1d(rollOff)]
    if len(ros) == 1:
        ros = ros * n_var
    if len(ros) != n_var:
        raise ValueError(f"rollOff must be one value or {n_var} of them (got {len(ros)})")
    return ros


def run_sim_mc_multi_adaptive(ensemble_max, cpLength, csLength, tailTx, tailRx, windowTx, windowRx, channel, snr, offset,
                              prefixRemovalLength, circularShiftLength, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff,
                              target_bit_errors, first_block=1, seed=0, handle=None):
    """run_sim_mc_adaptive for n_var configurations on the same symbols in one call
    (Handle.ber_run_masked_adaptive_multi): windowTx and windowRx are lists of n_var (diagonal matrices or vectors),
    rollOff one integer or n_var of them.  Configuration v's unmasked chain has noise stream v, its masked chain n_var + v,
    as in run_sim_mc_multi; every SNR point runs until all 2 n_var chains have counted target_bit_errors bit errors, or
    ensemble_max ensemble indices.  Returns (berMasked, ber, ensemble_used) of shapes (n_var, n_snr), (n_var, n_snr) and
    (n_snr,); with one configuration this is run_sim_mc_adaptive's result exactly."""
    wts, wrs = list(windowTx), list(windowRx)
    if len(wts) != len(wrs) or not wts:
        raise ValueError(f"windowTx and windowRx must be lists of the same length (got {len(wts)}, {len(wrs)})")
    ros = _roll_off_list(rollOff, len(wts))
    h = handle or default_handle()
    s = capi.SysT(N=int(numSubcar), cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), tail_rx=int(tailRx),
                  rm=int(prefixRemovalLength), shift=int(circularShiftLength), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    ch = np.atleast_2d(np.asarray(channel)).T                         # (L, C)
    r = h.ber_run_masked_adaptive_multi(s, [_diag(w) for w in wts], [_diag(w) for w in wrs], ch,
                                        np.atleast_1d(np.asarray(snr, dtype=np.float64)), int(ensemble_max),
                                        target_bit_errors=int(target_bit_errors), first_block=int(first_block), seed=seed,
                                        variant=0, roll_offs=ros)
    return r["bit_err"][0] / r["bit_tot"], r["bit_err"][1] / r["bit_tot"], r["ensemble_used"]


def obr_split(x, offset):
    """(obr, mf_band) of an 8N-point fftshifted PSD of a guard-band signal: the guard band is the first and the last
    8*offset bins (8x interpolation), its mean the out-of-band radiation; mf_band the bins in between."""
    gb = 8 * int(offset)
    if gb < 1 or 2 * gb >= len(x):
        raise ValueError("the OBR needs 1 <= offset < numSubcar/2")
    return float(np.mean(np.hstack((x[:gb], x[-gb:])))), x[gb:len(x) - gb]


def psd_sim_mc(numFrames, cpLength, csLength, tailTx, windowTx, offset, numSubcar, bitsPerSubcar, symbolsPerTx, rollOff,
               seed=0, estimator="reference", handle=None):
    """PSD of the Tx signal of run_sim_mc (matlab/main_channel_mask.m:334-431) with and without the DFT-domain
    raised-cosine mask, on frames 0 .. numFrames-1 of run_sim_mc's draws with the same seed (Handle.psd_masked).
    MATLAB conventions (Gray unit-power QAM), guard = offset; windowTx a diagonal matrix or a vector.  estimator:
    "reference" (__psd_estimate's slices) or "hann" (sin^2 taper, 50 % overlap).  Returns estimate_obr-style keys:
    X_est_masked / X_est (8N bins, fftshifted), obr_masked / obr (mean over the guard band), mf_band_masked / mf_band (the
    bins in between) and f_axis in cycles per sample."""
    if int(offset) < 1:
        raise ValueError("the OBR needs offset >= 1")
    h = handle or default_handle()
    N = int(numSubcar)
    s = capi.SysT(N=N, cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    xm, xu = h.psd_masked(s, _diag(windowTx), roll_off=int(rollOff), frames=int(numFrames), seed=seed, estimator=estimator)
    out = {"X_est_masked": xm, "X_est": xu, "f_axis": np.linspace(-.5, .5 - 1 / (8 * N), 8 * N)}
    out["obr_masked"], out["mf_band_masked"] = obr_split(xm, offset)
    out["obr"], out["mf_band"] = obr_split(xu, offset)
    return out


def psd_sim_mc_multi(numFrames, cpLength, csLength, tailTx, windowTx, offset, numSubcar, bitsPerSubcar, symbolsPerTx,
                     rollOff, seed=0, estimator="reference", handle=None):
    """psd_sim_mc for n_var configurations on the same frames in one call (Handle.psd_masked_multi): windowTx a list of
    n_var Tx windows (diagonal matrices or vectors), rollOff one integer or n_var of them.  The same keys as psd_sim_mc,
    one row per configuration: X_est_masked / X_est (n_var, 8N), obr_masked / obr (n_var,), mf_band_masked / mf_band
    (n_var, 8N - 16 offset), and f_axis.  With one configuration it equals psd_sim_mc up to the order of fp64 additions."""
    if int(offset) < 1:
        raise ValueError("the OBR needs offset >= 1")
    wts = list(windowTx)
    if not wts:
        raise ValueError("windowTx must be a non-empty list")
    ros = _roll_off_list(rollOff, len(wts))
    h = handle or default_handle()
    N = int(numSubcar)
    s = capi.SysT(N=N, cp=int(cpLength), cs=int(csLength), tail_tx=int(tailTx), bits=int(bitsPerSubcar),
                  S=int(symbolsPerTx), noise_norm=1, constellation=1, precision=0, guard=int(offset))
    xm, xu = h.psd_masked_multi(s, [_diag(w) for w in wts], roll_offs=ros, frames=int(numFrames), seed=seed,
                                estimator=estimator)
    out = {"X_est_masked": xm, "X_est": xu, "f_axis": np.linspace(-.5, .5 - 1 / (8 * N), 8 * N)}
    for key, x in (("masked", xm), ("", xu)):
        parts = [obr_split(row, offset) for row in x]
        sfx = "_" + key if key else ""
        out["obr" + sfx] = np.array([p[0] for p in parts])
        out["mf_band" + sfx] = np.stack([p[1] for p in parts])
    return out


def calculate_interference(cpLength, typeOFDM, windowTx, windowRx, numSubcar, tailTx, tailRx, channels, mode=0,
                           handle=None):
    """Scalar interference power on the mean of `channels` (rows = realisations, as vehA200channel2 is stored),
    matlab/main_interference_calculation.m:177-225; settings are passed explicitly instead of settingsData.mat."""
    h = handle or default_handle()
    s = capi.params_from_name(typeOFDM, int(numSubcar), int(cpLength), int(tailTx), int(tailRx))
    mean_ir = np.asarray(channels).mean(axis=0)                       # :196
    return float(h.interf_power(s, _diag(windowTx), _diag(windowRx), mean_ir[:, None], mode=mode, scalar=True)[0])


def _quad_objective(side, typeOFDM, window_fixed, numSubcar, cpLength, tailTx, tailRx, channel, alpha, handle=None,
                    channel_set=False):
    """channel_set: `channel` is an (L, C) set and the parts are its means (wofdm_window_hessian_parts_set); the result is
    linear in the parts, so it is the mean of the per-channel quad_objective."""
    h = handle or default_handle()
    s = capi.params_from_name(typeOFDM, int(numSubcar), int(cpLength), int(tailTx), int(tailRx))
    fixed = _diag(window_fixed)
    parts = h.window_hessian_parts_set if channel_set else h.window_hessian_parts
    if side == "tx":
        Hc, Hs = parts(s, channel, np.eye(s.n_tx), fixed[None, :])
    else:
        Hc, Hs = parts(s, channel, fixed[None, :], np.eye(s.N + s.tail_rx))
    return float(alpha) * Hc + (1.0 - float(alpha)) * np.diag(Hs.sum(axis=1))


def quad_objective_tx(windowRx, numSubcar, tailRx, cpLength, typeOFDM, tailTx, channel, alpha, handle=None):
    """HTx of quad_objective_tx (matlab/window_optimization.m:596-634): the full Tx window (n_tx entries) is the variable,
    windowRx (diagonal matrix or vector) is fixed; H = 2 (alpha H1 + (1 - alpha) H2) with H1 the off-diagonal ICI term and
    H2 = real(diag(diag(B2' B2 C C'))) (:628-631).  The script hands over array_ici_isi of the mean channel
    (:224-229); here `channel` is that impulse response and the device builds the matrices; prefixRemovalLength,
    circularShiftLength and csLength follow from calculate_parameters for typeOFDM."""
    return _quad_objective("tx", typeOFDM, windowRx, numSubcar, cpLength, tailTx, tailRx, channel, alpha, handle)


def quad_objective_rx(windowTx, numSubcar, tailRx, cpLength, typeOFDM, tailTx, channel, alpha, handle=None):
    """HRx of quad_objective_rx (matlab/window_optimization.m:637-680): the full Rx window (N + tailRx entries) is the
    variable, windowTx is fixed."""
    return _quad_objective("rx", typeOFDM, windowTx, numSubcar, cpLength, tailTx, tailRx, channel, alpha, handle)


def quad_objective_tx_expected(windowRx, numSubcar, tailRx, cpLength, typeOFDM, tailTx, channels, alpha, handle=None):
    """quad_objective_tx averaged over a channel set: `channels` is C x L, rows = realisations (as vehA200channel2 is
    stored), and the result is the mean over the rows of quad_objective_tx -- the expected interference instead of the
    interference of the mean channel."""
    ch = np.atleast_2d(np.asarray(channels)).T
    return _quad_objective("tx", typeOFDM, windowRx, numSubcar, cpLength, tailTx, tailRx, ch, alpha, handle, channel_set=True)


def quad_objective_rx_expected(windowTx, numSubcar, tailRx, cpLength, typeOFDM, tailTx, channels, alpha, handle=None):
    """quad_objective_rx averaged over a channel set (`channels` C x L, rows = realisations)."""
    ch = np.atleast_2d(np.asarray(channels)).T
    return _quad_objective("rx", typeOFDM, windowTx, numSubcar, cpLength, tailTx, tailRx, ch, alpha, handle, channel_set=True)
