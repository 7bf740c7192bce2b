"""ctypes binding of libwofdm.so (include/wofdm.h).

The library is the product; this file only marshals numpy arrays into the C-ABI.  There is no
CPU fallback: importing works anywhere (so host logic and symbol exports can be tested), but
creating a handle without a CUDA device raises ``WofdmError``.
"""
from __future__ import annotations

import ctypes as C
import weakref
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwofdm.so")

OK, EINVAL, ECUDA, ENOMEM, ENODEV, EUNSUPPORTED = 0, -1, -2, -3, -4, -5
WOFDM_BY_SUBCARRIER, WOFDM_BY_CHANNEL = 1, 2         # wofdm_ber_run_resolved: resolve flags
WOFDM_TARGET_BIT_ERRORS, WOFDM_TARGET_SYMBOL_ERRORS = 0, 1   # wofdm_ber_run_adaptive: target_kind
_ERRNAME = {EINVAL: "WOFDM_EINVAL", ECUDA: "WOFDM_ECUDA", ENOMEM: "WOFDM_ENOMEM", ENODEV: "WOFDM_ENODEV",
            EUNSUPPORTED: "WOFDM_EUNSUPPORTED"}


class WofdmError(RuntimeError):
    def __init__(self, code, msg=""):
        self.code = code
        super().__init__(f"{_ERRNAME.get(code, code)}: {msg}")


class SysT(C.Structure):
    """wofdm_sys_t"""
    _fields_ = [(n, C.c_int32) for n in ("N", "cp", "cs", "tail_tx", "tail_rx", "rm", "shift", "bits", "S",
                                         "noise_norm", "constellation", "precision", "guard")]

    @property
    def n_active(self):
        return self.N - 2 * self.guard

    @property
    def n_tx(self):
        return self.N + self.cp + self.cs

    @property
    def stride(self):
        return self.n_tx - self.tail_tx

    def noise_len(self, L):
        return self.S * self.stride if self.noise_norm == 0 else self.tail_tx + self.S * self.stride + L - 1

    def copy(self, **kw):
        o = SysT()
        C.memmove(C.byref(o), C.byref(self), C.sizeof(SysT))
        for k, v in kw.items():
            setattr(o, k, v)
        return o


_P = C.POINTER
_dp, _i32p, _i64p = _P(C.c_double), _P(C.c_int32), _P(C.c_int64)
# wofdm_reduce_fn: int (*)(int64_t* counts, int64_t n, void* user)
REDUCE_FN = C.CFUNCTYPE(C.c_int, _i64p, C.c_int64, C.c_void_p)

# name -> (restype, argtypes); every symbol include/wofdm.h declares
SIGNATURES = {
    "wofdm_version": (C.c_int, []),
    "wofdm_device_count": (C.c_int, [_P(C.c_int)]),
    "wofdm_create": (C.c_int, [_P(C.c_void_p), C.c_int]),
    "wofdm_create_on": (C.c_int, [_P(C.c_void_p), _P(C.c_int), C.c_int]),
    "wofdm_destroy": (C.c_int, [C.c_void_p]),
    "wofdm_last_error": (C.c_char_p, [C.c_void_p]),
    "wofdm_launch_count": (C.c_int64, [C.c_void_p]),
    "wofdm_diag_fp32_peak": (C.c_int, [C.c_void_p, C.c_int, _dp, _dp]),
    "wofdm_params_from_name": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, _P(SysT)]),
    "wofdm_rc_window_tx": (C.c_int, [_P(SysT), _dp]),
    "wofdm_rc_window_rx": (C.c_int, [_P(SysT), _dp]),
    "wofdm_expand_window_tx": (C.c_int, [_P(SysT), _dp, _dp]),
    "wofdm_expand_window_rx": (C.c_int, [_P(SysT), _dp, _dp]),
    "wofdm_ber_run": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                C.c_uint64, C.c_uint32, _i64p, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_shard": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                      C.c_uint64, C.c_uint32, C.c_int, C.c_int, _i64p, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_multi": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                      C.c_uint64, C.c_uint32, C.c_int, C.c_int, _i64p, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_resolved": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                         C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_segments": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                         _i64p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_adaptive": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                         C.c_int64, C.c_int, C.c_int64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, REDUCE_FN,
                                         C.c_void_p, _i64p, _i64p, _i64p, _i64p, _i64p, _P(C.c_int)]),
    "wofdm_ber_plan_create_multi": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, C.c_int, _dp, C.c_int, C.c_int, _dp, C.c_int,
                                              _P(C.c_void_p)]),
    "wofdm_ber_plan_variants": (C.c_int, [C.c_void_p, _P(C.c_int)]),
    "wofdm_ber_plan_create": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int,
                                        _P(C.c_void_p)]),
    "wofdm_ber_plan_launch": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_uint32, C.c_int, C.c_int,
                                        C.c_void_p, _P(C.c_void_p)]),
    "wofdm_ber_plan_read": (C.c_int, [C.c_void_p, _i64p, _i64p]),
    "wofdm_ber_plan_kernel": (C.c_char_p, [C.c_void_p]),
    "wofdm_ber_plan_destroy": (C.c_int, [C.c_void_p]),
    "wofdm_ber_verify": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, _i32p, _dp, C.c_int,
                                   _dp, _i32p, _i64p, _i64p]),
    "wofdm_ber_draws": (C.c_int, [C.c_void_p, _P(SysT), C.c_int, C.c_uint64, C.c_uint32, _i64p, C.c_int, _i32p, _dp]),
    "wofdm_interf_power": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, C.c_int, _dp]),
    "wofdm_interf_power_scalar": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, C.c_int, _dp]),
    "wofdm_interf_last_timing": (C.c_int, [C.c_void_p, _dp, _dp, _dp, _P(C.c_int), _P(C.c_int)]),
    "wofdm_ber_run_masked": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64, C.c_uint64,
                                       C.c_uint32, C.c_int, _i64p, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_masked_shard": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                             C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, _i64p, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_masked_multi": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _P(C.c_int), C.c_int, _dp, C.c_int, C.c_int, _dp,
                                             C.c_int, C.c_int64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, _i64p, _i64p, _i64p,
                                             _i64p]),
    "wofdm_ber_run_masked_resolved": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                                C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_masked_segments": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                                _i64p, C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int,
                                                _i64p, _i64p, _i64p]),
    "wofdm_ber_run_masked_adaptive": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _dp, C.c_int, C.c_int, _dp, C.c_int, C.c_int64,
                                                C.c_int64, C.c_int, C.c_int64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int,
                                                REDUCE_FN, C.c_void_p, _i64p, _i64p, _i64p, _i64p, _i64p, _P(C.c_int)]),
    "wofdm_ber_run_masked_segments_multi": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _P(C.c_int), C.c_int, _dp, C.c_int,
                                                      C.c_int, _dp, C.c_int, C.c_int64, _i64p, C.c_int, C.c_uint64, C.c_uint32,
                                                      C.c_int, C.c_int, C.c_int, _i64p, _i64p, _i64p]),
    "wofdm_ber_run_masked_adaptive_multi": (C.c_int, [C.c_void_p, _P(SysT), _dp, _dp, _P(C.c_int), C.c_int, _dp, C.c_int,
                                                      C.c_int, _dp, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int64,
                                                      C.c_uint64, C.c_uint32, C.c_int, C.c_int, REDUCE_FN, C.c_void_p, _i64p,
                                                      _i64p, _i64p, _i64p, _i64p, _P(C.c_int)]),
    "wofdm_window_hessian": (C.c_int, [C.c_void_p, _P(SysT), _dp, C.c_int, _dp, _P(C.c_int)]),
    "wofdm_window_hessian_parts": (C.c_int, [C.c_void_p, _P(SysT), _dp, C.c_int, _dp, C.c_int, _dp, C.c_int, _dp, _dp]),
    "wofdm_window_hessian_set": (C.c_int, [C.c_void_p, _P(SysT), _dp, C.c_int, C.c_int, _dp, _P(C.c_int)]),
    "wofdm_window_hessian_parts_set": (C.c_int, [C.c_void_p, _P(SysT), _dp, C.c_int, C.c_int, _dp, C.c_int, _dp, C.c_int,
                                                 _dp, _dp]),
    "wofdm_window_hessian_last_timing": (C.c_int, [C.c_void_p, _dp, _dp, _P(C.c_int)]),
    "wofdm_channel_profile": (C.c_int, [C.c_char_p]),
    "wofdm_gen_channels": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                     C.c_uint64, _dp, _dp]),
    "wofdm_psd_estimate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_int, C.c_int,
                                     C.c_int64, C.c_uint64, _i32p, _dp]),
    "wofdm_psd_masked": (C.c_int, [C.c_void_p, _P(SysT), _dp, C.c_int, C.c_uint64, C.c_int64, C.c_int64, C.c_int, _dp, _dp]),
    "wofdm_psd_masked_multi": (C.c_int, [C.c_void_p, _P(SysT), _dp, _P(C.c_int), C.c_int, C.c_uint64, C.c_int64, C.c_int64,
                                         C.c_int, _dp, _dp]),
}

_lib = None


def load():
    """dlopen libwofdm.so (built by ``__graft_entry__.build()`` / ``make -C csrc``)."""
    global _lib
    if _lib is None:
        path = os.environ.get("WOFDM_LIB", LIB_PATH)       # development aid: an alternative build of the same library
        if not os.path.exists(path):
            raise WofdmError(ENODEV, f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; "
                                     f"g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _cplx(a):
    """complex array -> contiguous complex128 (interleaved re, im doubles)"""
    return np.ascontiguousarray(a, dtype=np.complex128)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def params_from_name(name, N, cp, tail_tx, tail_rx, bits=4, S=16, noise_norm=0, constellation=0, precision=0, guard=0):
    s = SysT(bits=bits, S=S, noise_norm=noise_norm, constellation=constellation, precision=precision, guard=guard)
    rc = load().wofdm_params_from_name(name.encode(), N, cp, tail_tx, tail_rx, C.byref(s))
    if rc:
        raise WofdmError(rc, f"unknown system {name!r}")
    return s


def rc_window_tx(s):
    out = np.empty(s.n_tx)
    rc = load().wofdm_rc_window_tx(C.byref(s), _ptr(out, _dp))
    if rc:
        raise WofdmError(rc, "rc_window_tx")
    return out


def rc_window_rx(s):
    out = np.empty(s.N + s.tail_rx)
    rc = load().wofdm_rc_window_rx(C.byref(s), _ptr(out, _dp))
    if rc:
        raise WofdmError(rc, "rc_window_rx")
    return out


def expand_window_tx(s, x):
    x = _f64(np.ravel(x))
    if x.size != s.tail_tx + 1:
        raise WofdmError(EINVAL, "Tx tail vector must hold tail_tx+1 values")
    out = np.empty(s.n_tx)
    rc = load().wofdm_expand_window_tx(C.byref(s), _ptr(x, _dp), _ptr(out, _dp))
    if rc:
        raise WofdmError(rc, "expand_window_tx")
    return out


def expand_window_rx(s, x):
    x = _f64(np.ravel(x))
    if x.size != s.tail_rx // 2 + 1:
        raise WofdmError(EINVAL, "Rx tail vector must hold tail_rx/2+1 values")
    out = np.empty(s.N + s.tail_rx)
    rc = load().wofdm_expand_window_rx(C.byref(s), _ptr(x, _dp), _ptr(out, _dp))
    if rc:
        raise WofdmError(rc, "expand_window_rx")
    return out


class Handle:
    """wofdm_handle.  devices: None = all visible, int n = first n, list = explicit ids."""

    def __init__(self, devices=None):
        lib = load()
        self._h = C.c_void_p()
        if devices is None or isinstance(devices, int):
            rc = lib.wofdm_create(C.byref(self._h), 0 if devices is None else int(devices))
        else:
            ids = (C.c_int * len(devices))(*devices)
            rc = lib.wofdm_create_on(C.byref(self._h), ids, len(devices))
        if rc:
            self._h = None
            raise WofdmError(rc, "wofdm_create failed (no CUDA device? this library has no CPU path)")
        self._plans = weakref.WeakSet()         # live BerPlan objects: a plan's native side points into this context

    def close(self):
        if getattr(self, "_h", None):
            for p in list(getattr(self, "_plans", ())):     # plans first: wofdm_ber_plan_destroy reads the context
                p.close()
            load().wofdm_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc, reduce_cb=None):
        if rc and getattr(reduce_cb, "error", None) is not None:      # the call failed because its reduce callback raised
            raise WofdmError(rc, f"reduce callback raised {reduce_cb.error!r}") from reduce_cb.error
        if rc:
            raise WofdmError(rc, (load().wofdm_last_error(self._h) or b"").decode())

    @property
    def launches(self):
        return int(load().wofdm_launch_count(self._h))

    def fp32_peak(self, mode=0):
        """(TFLOP/s, equivalent SM MHz) of the FMA-only micro-benchmark (0 scalar FFMA, 1 FFMA2)."""
        t, m = C.c_double(), C.c_double()
        self._check(load().wofdm_diag_fp32_peak(self._h, int(mode), C.byref(t), C.byref(m)))
        return t.value, m.value

    # ---- BER ----
    def _win_chan(self, s, win_tx, win_rx, chan):
        wt, wr = _f64(np.ravel(win_tx)), _f64(np.ravel(win_rx))
        if wt.size != s.n_tx or wr.size != s.N + s.tail_rx:
            raise WofdmError(EINVAL, f"window sizes must be n_tx={s.n_tx} and N+tail_rx={s.N + s.tail_rx}")
        ch = np.asarray(chan)
        if ch.ndim == 1:
            ch = ch[:, None]
        L, Cn = ch.shape
        chf = _cplx(ch.T)          # (C, L) row-major == L x C column-major
        return wt, wr, chf, L, Cn

    def ber_run(self, s, win_tx, win_rx, chan, snr_db, ensemble, seed=0, variant=0, shard=(0, 1)):
        wt, wr, chf, L, Cn = self._win_chan(s, win_tx, win_rx, chan)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        out = [np.zeros(n, dtype=np.int64) for _ in range(4)]
        rc = load().wofdm_ber_run_shard(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, Cn,
                                        _ptr(snr, _dp), n, int(ensemble), int(seed), int(variant),
                                        int(shard[0]), int(shard[1]), *[_ptr(o, _i64p) for o in out])
        self._check(rc)
        return dict(bit_err=out[0], bit_tot=out[1], sym_err=out[2], sym_tot=out[3])

    def _win_multi(self, s, wins_tx, wins_rx):
        """(n_var, n_tx), (n_var, N+tail_rx) contiguous doubles from lists / 2-D arrays of windows."""
        wt = _f64(np.atleast_2d(np.asarray(wins_tx, dtype=np.float64)))
        wr = _f64(np.atleast_2d(np.asarray(wins_rx, dtype=np.float64)))
        if wt.ndim != 2 or wr.ndim != 2 or wt.shape[0] != wr.shape[0] or wt.shape[1] != s.n_tx or wr.shape[1] != s.N + s.tail_rx:
            raise WofdmError(EINVAL, f"windows must be (n_var, n_tx={s.n_tx}) and (n_var, N+tail_rx={s.N + s.tail_rx})")
        return wt, wr

    def ber_run_multi(self, s, wins_tx, wins_rx, chan, snr_db, ensemble, seed=0, variant=0, shard=(0, 1)):
        """n_var window pairs on the same symbols (wofdm_ber_run_multi).  bit_err / sym_err: (n_var, n_snr);
        pair v = ber_run(..., variant=variant + v) with its windows."""
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        snr = _f64(np.ravel(snr_db))
        n, nv = snr.size, wt.shape[0]
        be, se = np.zeros((nv, n), dtype=np.int64), np.zeros((nv, n), dtype=np.int64)
        bt, st = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
        rc = load().wofdm_ber_run_multi(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), nv, _ptr(chf, _dp), L, Cn,
                                        _ptr(snr, _dp), n, int(ensemble), int(seed), int(variant), int(shard[0]), int(shard[1]),
                                        _ptr(be, _i64p), _ptr(bt, _i64p), _ptr(se, _i64p), _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, bit_tot=bt, sym_err=se, sym_tot=st)

    def ber_run_resolved(self, s, wins_tx, wins_rx, chan, snr_db, ensemble, seed=0, variant=0, shard=(0, 1),
                         by_subcarrier=True, by_channel=False):
        """ber_run_multi with the counters resolved by sub-carrier and / or channel (wofdm_ber_run_resolved).
        bit_err / sym_err: (n_var, n_snr, Cr, Nr), sym_tot / bit_tot: (n_snr, Cr, Nr), Cr = C if by_channel else 1,
        Nr = N (FFT bin order) if by_subcarrier else 1.  Summed over the last two axes: ber_run_multi's counters."""
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        snr = _f64(np.ravel(snr_db))
        n, nv = snr.size, wt.shape[0]
        resolve, shape = _resolve(s, n, Cn, by_subcarrier, by_channel)
        be, se = np.zeros((nv,) + shape, dtype=np.int64), np.zeros((nv,) + shape, dtype=np.int64)
        st = np.zeros(shape, dtype=np.int64)
        rc = load().wofdm_ber_run_resolved(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), nv, _ptr(chf, _dp), L, Cn,
                                           _ptr(snr, _dp), n, int(ensemble), int(seed), int(variant), int(shard[0]),
                                           int(shard[1]), int(resolve), _ptr(be, _i64p), _ptr(se, _i64p), _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, sym_err=se, sym_tot=st, bit_tot=st * int(s.bits))

    def ber_run_segments(self, s, wins_tx, wins_rx, chan, snr_db, ensemble_max, segments, seed=0, variant=0, shard=(0, 1),
                         by_subcarrier=False, by_channel=False):
        """A chosen subset of a job's frames (wofdm_ber_run_segments).  segments: (n_seg, 3) {snr_idx, e_begin, e_count}, every
        channel of point snr_idx at ensemble indices [e_begin, e_begin + e_count) of a job of ensemble_max indices; frames and
        draws are those of ber_run_multi(..., ensemble=ensemble_max).  Unresolved: bit_err / sym_err (n_var, n_snr), sym_tot /
        bit_tot (n_snr,); resolved: the shapes of ber_run_resolved."""
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        snr = _f64(np.ravel(snr_db))
        n, nv = snr.size, wt.shape[0]
        seg = np.ascontiguousarray(np.asarray(segments, dtype=np.int64).reshape(-1, 3))
        resolve, shape = _resolve(s, n, Cn, by_subcarrier, by_channel)
        be, se = np.zeros((nv,) + shape, dtype=np.int64), np.zeros((nv,) + shape, dtype=np.int64)
        st = np.zeros(shape, dtype=np.int64)
        rc = load().wofdm_ber_run_segments(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), nv, _ptr(chf, _dp), L, Cn,
                                           _ptr(snr, _dp), n, int(ensemble_max), _ptr(seg, _i64p), seg.shape[0], int(seed),
                                           int(variant), int(shard[0]), int(shard[1]), int(resolve),
                                           _ptr(be, _i64p), _ptr(se, _i64p), _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, sym_err=se, sym_tot=st, bit_tot=st * int(s.bits))

    def ber_run_adaptive(self, s, wins_tx, wins_rx, chan, snr_db, ensemble_max, target_bit_errors=None,
                         target_symbol_errors=None, first_block=1, seed=0, variant=0, shard=(0, 1), reduce=None):
        """Run every SNR point until the fewest errors over the window pairs reach the target, or to ensemble_max ensemble
        indices (wofdm_ber_run_adaptive; the schedule is stated in include/wofdm.h).  Exactly one of target_bit_errors /
        target_symbol_errors.  reduce: None, or a callable on this process's round counts, an int64 array (n_var, n_snr, 2)
        of {bit, sym}, that returns (or fills in place) their sum over the processes -- sharding.adaptive_allreduce() under
        torch.distributed.  Returns bit_err / sym_err (n_var, n_snr), bit_tot / sym_tot (n_snr,), ensemble_used (n_snr,)
        and rounds."""
        kind, target = _target(target_bit_errors, target_symbol_errors)
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        snr = _f64(np.ravel(snr_db))
        n, nv = snr.size, wt.shape[0]
        be, se = np.zeros((nv, n), dtype=np.int64), np.zeros((nv, n), dtype=np.int64)
        bt, st, used = (np.zeros(n, dtype=np.int64) for _ in range(3))
        rounds = C.c_int(0)
        cb = reduce_trampoline(reduce, (nv, n, 2)) if reduce is not None else REDUCE_FN()
        rc = load().wofdm_ber_run_adaptive(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), nv, _ptr(chf, _dp), L, Cn,
                                           _ptr(snr, _dp), n, int(ensemble_max), int(first_block), kind, int(target), int(seed),
                                           int(variant), int(shard[0]), int(shard[1]), cb, None, _ptr(used, _i64p),
                                           _ptr(be, _i64p), _ptr(bt, _i64p), _ptr(se, _i64p), _ptr(st, _i64p), C.byref(rounds))
        self._check(rc, cb)
        return dict(bit_err=be, bit_tot=bt, sym_err=se, sym_tot=st, ensemble_used=used, rounds=rounds.value)

    def ber_run_masked(self, s, win_tx, win_rx, chan, snr_db, ensemble, seed=0, variant=0, roll_off=10, shard=(0, 1)):
        """Channel-mask variant (wofdm_ber_run_masked_shard): counters of the MASKED signal; ber_run with the same `s`
        (s.guard = the script's offset) gives the unmasked ones on the same symbols.  shard=(k, W): the k-th of W
        contiguous blocks of the frame ids (not f = k mod W as in ber_run); the W shards add up to (0, 1)."""
        wt, wr, chf, L, Cn = self._win_chan(s, win_tx, win_rx, chan)
        snr = _f64(np.ravel(snr_db))
        out = [np.zeros(snr.size, dtype=np.int64) for _ in range(4)]
        rc = load().wofdm_ber_run_masked_shard(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, Cn,
                                               _ptr(snr, _dp), snr.size, int(ensemble), int(seed), int(variant), int(roll_off),
                                               int(shard[0]), int(shard[1]), *[_ptr(o, _i64p) for o in out])
        self._check(rc)
        return dict(bit_err=out[0], bit_tot=out[1], sym_err=out[2], sym_tot=out[3])

    def ber_run_masked_multi(self, s, wins_tx, wins_rx, chan, snr_db, ensemble, seed=0, variant=0, roll_offs=10, shard=(0, 1)):
        """n_var window pairs of the channel-mask chain on the same frames (wofdm_ber_run_masked_multi): pair v = ber_run_masked(
        ..., variant=variant + v, roll_off=roll_offs[v], shard=shard) with its windows, bit for bit.  roll_offs: one value for
        every pair, or n_var values.  bit_err / sym_err: (n_var, n_snr); bit_tot / sym_tot: (n_snr,)."""
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        nv = wt.shape[0]
        ro = _roll_offs(roll_offs, nv)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        be, se = np.zeros((nv, n), dtype=np.int64), np.zeros((nv, n), dtype=np.int64)
        bt, st = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int64)
        rc = load().wofdm_ber_run_masked_multi(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(ro, _P(C.c_int)), nv,
                                               _ptr(chf, _dp), L, Cn, _ptr(snr, _dp), n, int(ensemble), int(seed), int(variant),
                                               int(shard[0]), int(shard[1]), _ptr(be, _i64p), _ptr(bt, _i64p), _ptr(se, _i64p),
                                               _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, bit_tot=bt, sym_err=se, sym_tot=st)

    def ber_run_masked_resolved(self, s, win_tx, win_rx, chan, snr_db, ensemble, seed=0, variant=0, roll_off=10, shard=(0, 1),
                                by_subcarrier=True, by_channel=False):
        """ber_run_masked with the counters resolved by sub-carrier and / or channel (wofdm_ber_run_masked_resolved).
        bit_err / sym_err / sym_tot / bit_tot: (n_snr, Cr, Nr), Cr = C if by_channel else 1, Nr = N (FFT bin order) if
        by_subcarrier else 1.  Summed over the last two axes: ber_run_masked's counters of the same shard."""
        wt, wr, chf, L, Cn = self._win_chan(s, win_tx, win_rx, chan)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        resolve, shape = _resolve(s, n, Cn, by_subcarrier, by_channel)
        be, se, st = (np.zeros(shape, dtype=np.int64) for _ in range(3))
        rc = load().wofdm_ber_run_masked_resolved(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, Cn,
                                                  _ptr(snr, _dp), n, int(ensemble), int(seed), int(variant), int(roll_off),
                                                  int(shard[0]), int(shard[1]), int(resolve),
                                                  _ptr(be, _i64p), _ptr(se, _i64p), _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, sym_err=se, sym_tot=st, bit_tot=st * int(s.bits))

    def ber_run_masked_segments(self, s, win_tx, win_rx, chan, snr_db, ensemble_max, segments, seed=0, variant=0, roll_off=10,
                                shard=(0, 1), by_subcarrier=False, by_channel=False):
        """A chosen subset of a masked job's frames (wofdm_ber_run_masked_segments).  segments: (n_seg, 3) {snr_idx, e_begin,
        e_count}, as in ber_run_segments; frames and draws are those of ber_run_masked(..., ensemble=ensemble_max).
        shard=(k, W): the k-th of W contiguous blocks of the local indices.  Unresolved: bit_err / sym_err / sym_tot / bit_tot
        (n_snr,); resolved: the (n_snr, Cr, Nr) shapes of ber_run_masked_resolved."""
        wt, wr, chf, L, Cn = self._win_chan(s, win_tx, win_rx, chan)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        seg = np.ascontiguousarray(np.asarray(segments, dtype=np.int64).reshape(-1, 3))
        resolve, shape = _resolve(s, n, Cn, by_subcarrier, by_channel)
        be, se, st = (np.zeros(shape, dtype=np.int64) for _ in range(3))
        rc = load().wofdm_ber_run_masked_segments(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, Cn,
                                                  _ptr(snr, _dp), n, int(ensemble_max), _ptr(seg, _i64p), seg.shape[0],
                                                  int(seed), int(variant), int(roll_off), int(shard[0]), int(shard[1]),
                                                  int(resolve), _ptr(be, _i64p), _ptr(se, _i64p), _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, sym_err=se, sym_tot=st, bit_tot=st * int(s.bits))

    def ber_run_masked_adaptive(self, s, win_tx, win_rx, chan, snr_db, ensemble_max, target_bit_errors=None,
                                target_symbol_errors=None, first_block=1, seed=0, variant=0, roll_off=10, shard=(0, 1),
                                reduce=None):
        """run_sim_mc with the stopping rule (wofdm_ber_run_masked_adaptive): the masked chain (row 0, noise stream
        variant + 1) and the unmasked chain (row 1, noise stream variant) on the same frames, every SNR point run until both
        rows reach the target or ensemble_max ensemble indices.  Exactly one of target_bit_errors / target_symbol_errors.
        reduce: as in ber_run_adaptive, on int64 counts of shape (2, n_snr, 2).  Returns bit_err / sym_err (2, n_snr),
        bit_tot / sym_tot (n_snr,), ensemble_used (n_snr,) and rounds."""
        kind, target = _target(target_bit_errors, target_symbol_errors)
        wt, wr, chf, L, Cn = self._win_chan(s, win_tx, win_rx, chan)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        be, se = np.zeros((2, n), dtype=np.int64), np.zeros((2, n), dtype=np.int64)
        bt, st, used = (np.zeros(n, dtype=np.int64) for _ in range(3))
        rounds = C.c_int(0)
        cb = reduce_trampoline(reduce, (2, n, 2)) if reduce is not None else REDUCE_FN()
        rc = load().wofdm_ber_run_masked_adaptive(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, Cn,
                                                  _ptr(snr, _dp), n, int(ensemble_max), int(first_block), kind, int(target),
                                                  int(seed), int(variant), int(roll_off), int(shard[0]), int(shard[1]), cb, None,
                                                  _ptr(used, _i64p), _ptr(be, _i64p), _ptr(bt, _i64p), _ptr(se, _i64p),
                                                  _ptr(st, _i64p), C.byref(rounds))
        self._check(rc, cb)
        return dict(bit_err=be, bit_tot=bt, sym_err=se, sym_tot=st, ensemble_used=used, rounds=rounds.value)

    def ber_run_masked_segments_multi(self, s, wins_tx, wins_rx, chan, snr_db, ensemble_max, segments, seed=0, variant=0,
                                      roll_offs=10, shard=(0, 1), by_subcarrier=False, by_channel=False):
        """ber_run_masked_segments for n_var window pairs on the same frames (wofdm_ber_run_masked_segments_multi): pair v =
        ber_run_masked_segments(..., variant=variant + v, roll_off=roll_offs[v]) with its windows, bit for bit.  roll_offs:
        one value for every pair, or n_var values.  Unresolved: bit_err / sym_err (n_var, n_snr), sym_tot / bit_tot
        (n_snr,); resolved: bit_err / sym_err (n_var, n_snr, Cr, Nr), sym_tot / bit_tot (n_snr, Cr, Nr).  One segment
        (s, 0, E) per point gives the resolved counters of several pairs over a whole job of E ensemble indices."""
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        nv = wt.shape[0]
        ro = _roll_offs(roll_offs, nv)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        seg = np.ascontiguousarray(np.asarray(segments, dtype=np.int64).reshape(-1, 3))
        resolve, shape = _resolve(s, n, Cn, by_subcarrier, by_channel)
        be, se = np.zeros((nv,) + shape, dtype=np.int64), np.zeros((nv,) + shape, dtype=np.int64)
        st = np.zeros(shape, dtype=np.int64)
        rc = load().wofdm_ber_run_masked_segments_multi(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(ro, _P(C.c_int)),
                                                        nv, _ptr(chf, _dp), L, Cn, _ptr(snr, _dp), n, int(ensemble_max),
                                                        _ptr(seg, _i64p), seg.shape[0], int(seed), int(variant), int(shard[0]),
                                                        int(shard[1]), int(resolve), _ptr(be, _i64p), _ptr(se, _i64p),
                                                        _ptr(st, _i64p))
        self._check(rc)
        return dict(bit_err=be, sym_err=se, sym_tot=st, bit_tot=st * int(s.bits))

    def ber_run_masked_adaptive_multi(self, s, wins_tx, wins_rx, chan, snr_db, ensemble_max, target_bit_errors=None,
                                      target_symbol_errors=None, first_block=1, seed=0, variant=0, roll_offs=10, shard=(0, 1),
                                      reduce=None):
        """ber_run_masked_adaptive for n_var window pairs / roll-offs on the same frames
        (wofdm_ber_run_masked_adaptive_multi): bit_err / sym_err (2, n_var, n_snr), block 0 the masked chain of pair v
        (noise stream variant + n_var + v), block 1 its unmasked chain (variant + v); a point stops when all 2 n_var rows
        reach the target or at ensemble_max.  roll_offs: one value for every pair, or n_var values.  reduce: as in
        ber_run_adaptive, on int64 counts of shape (2, n_var, n_snr, 2).  Returns also bit_tot / sym_tot (n_snr,),
        ensemble_used (n_snr,) and rounds."""
        kind, target = _target(target_bit_errors, target_symbol_errors)
        wt, wr = self._win_multi(s, wins_tx, wins_rx)
        _, _, chf, L, Cn = self._win_chan(s, wt[0], wr[0], chan)
        nv = wt.shape[0]
        ro = _roll_offs(roll_offs, nv)
        snr = _f64(np.ravel(snr_db))
        n = snr.size
        be, se = np.zeros((2, nv, n), dtype=np.int64), np.zeros((2, nv, n), dtype=np.int64)
        bt, st, used = (np.zeros(n, dtype=np.int64) for _ in range(3))
        rounds = C.c_int(0)
        cb = reduce_trampoline(reduce, (2, nv, n, 2)) if reduce is not None else REDUCE_FN()
        rc = load().wofdm_ber_run_masked_adaptive_multi(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(ro, _P(C.c_int)),
                                                        nv, _ptr(chf, _dp), L, Cn, _ptr(snr, _dp), n, int(ensemble_max),
                                                        int(first_block), kind, int(target), int(seed), int(variant),
                                                        int(shard[0]), int(shard[1]), cb, None, _ptr(used, _i64p),
                                                        _ptr(be, _i64p), _ptr(bt, _i64p), _ptr(se, _i64p), _ptr(st, _i64p),
                                                        C.byref(rounds))
        self._check(rc, cb)
        return dict(bit_err=be, bit_tot=bt, sym_err=se, sym_tot=st, ensemble_used=used, rounds=rounds.value)

    def psd_estimate(self, N, cp, cs, tail_tx, win_tx, guard_band=48, n_sym=256, records=1, seed=0, sym_idx=None,
                     bits=4, constellation=0):
        """X_est of timefreq_simulation.py:104-123 for the Tx signal of window win_tx (8N doubles, fftshifted), averaged
        over `records` records; sym_idx (records, n_sym, N - 2*guard_band) injects the constellation indices."""
        w = _f64(np.ravel(win_tx))
        if w.size != N + cp + cs:
            raise WofdmError(EINVAL, "psd_estimate: win_tx must have N + cp + cs entries")
        si = None
        if sym_idx is not None:
            si = np.ascontiguousarray(sym_idx, dtype=np.int32)
            if si.shape != (records, n_sym, N - 2 * guard_band):
                raise WofdmError(EINVAL, "psd_estimate: sym_idx must be (records, n_sym, N - 2*guard_band)")
        out = np.empty(8 * N, dtype=np.float64)
        rc = load().wofdm_psd_estimate(self._h, N, cp, cs, tail_tx, bits, constellation, _ptr(w, _dp), guard_band, n_sym,
                                       records, seed, _ptr(si, _i32p) if si is not None else None, _ptr(out, _dp))
        self._check(rc)
        return out

    def psd_masked(self, s, win_tx, roll_off=10, frames=1, f0=0, seed=0, estimator="reference", masked=True, unmasked=True):
        """PSD of the channel-mask chain's Tx streams (wofdm_psd_masked): frames f0 .. f0 + frames - 1, the symbols
        ber_run_masked / ber_run give them with the same `s` and seed; estimator "reference" (__psd_estimate) or "hann"
        (sin^2 taper, 50 % overlap).  Returns (masked, unmasked), each 8N doubles (fftshifted) or None where not asked for."""
        w = _f64(np.ravel(win_tx))
        if w.size != s.n_tx:
            raise WofdmError(EINVAL, f"psd_masked: win_tx must have n_tx={s.n_tx} entries")
        est = {"reference": 0, "hann": 1}.get(estimator)
        if est is None:
            raise WofdmError(EINVAL, f"psd_masked: estimator must be 'reference' or 'hann', not {estimator!r}")
        om = np.empty(8 * s.N, dtype=np.float64) if masked else None
        ou = np.empty(8 * s.N, dtype=np.float64) if unmasked else None
        rc = load().wofdm_psd_masked(self._h, C.byref(s), _ptr(w, _dp), int(roll_off), int(seed), int(f0), int(frames), est,
                                     _ptr(om, _dp) if om is not None else None, _ptr(ou, _dp) if ou is not None else None)
        self._check(rc)
        return om, ou

    def psd_masked_multi(self, s, wins_tx, roll_offs=10, frames=1, f0=0, seed=0, estimator="reference", masked=True,
                         unmasked=True):
        """psd_masked for n_var Tx windows / roll-offs on the same frames (wofdm_psd_masked_multi): row v = psd_masked with
        window v and roll_offs[v], up to the order of fp64 additions; one symbol draw, one mask product and one PSD launch per
        batch for every spectrum.  roll_offs: one value for every window, or n_var values.  Returns (masked, unmasked), each
        (n_var, 8N) doubles (fftshifted) or None where not asked for."""
        w = _f64(np.atleast_2d(np.asarray(wins_tx, dtype=np.float64)))
        if w.ndim != 2 or w.shape[1] != s.n_tx:
            raise WofdmError(EINVAL, f"psd_masked_multi: windows must be (n_var, n_tx={s.n_tx})")
        nv = w.shape[0]
        ro = _roll_offs(roll_offs, nv)
        est = {"reference": 0, "hann": 1}.get(estimator)
        if est is None:
            raise WofdmError(EINVAL, f"psd_masked_multi: estimator must be 'reference' or 'hann', not {estimator!r}")
        om = np.empty((nv, 8 * s.N), dtype=np.float64) if masked else None
        ou = np.empty((nv, 8 * s.N), dtype=np.float64) if unmasked else None
        rc = load().wofdm_psd_masked_multi(self._h, C.byref(s), _ptr(w, _dp), _ptr(ro, _P(C.c_int)), nv, int(seed), int(f0),
                                           int(frames), est, _ptr(om, _dp) if om is not None else None,
                                           _ptr(ou, _dp) if ou is not None else None)
        self._check(rc)
        return om, ou

    def ber_plan_multi(self, s, wins_tx, wins_rx, chan, snr_db):
        """Device-resident plan of n_var window pairs (wofdm_ber_plan_create_multi)."""
        return BerPlan(self, s, wins_tx, wins_rx, chan, snr_db, multi=True)

    def ber_plan(self, s, win_tx, win_rx, chan, snr_db):
        return BerPlan(self, s, win_tx, win_rx, chan, snr_db)

    def ber_verify(self, s, win_tx, win_rx, chan, snr_db, sym_idx, noise, force_staged=False, direct=False, no_tconv=False):
        """chan (L, F); snr_db (F,); sym_idx (F, S, N) ints; noise (F, noise_len) complex.
        Returns eq (F, S-1, N) complex, dec (F, S-1, N) int32, bit_err (F,), sym_err (F,)."""
        wt, wr, chf, L, F = self._win_chan(s, win_tx, win_rx, chan)
        snr = _f64(np.ravel(snr_db))
        si = np.ascontiguousarray(sym_idx, dtype=np.int32)
        nz = _cplx(noise)
        if snr.size != F or si.shape != (F, s.S, s.N) or nz.shape != (F, s.noise_len(L)):
            raise WofdmError(EINVAL, "verify: inconsistent shapes")
        eq = np.empty((F, s.S - 1, s.N), dtype=np.complex128)
        dec = np.empty((F, s.S - 1, s.N), dtype=np.int32)
        be, se = np.zeros(F, dtype=np.int64), np.zeros(F, dtype=np.int64)
        rc = load().wofdm_ber_verify(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, F,
                                     _ptr(snr, _dp), _ptr(si, _i32p), _ptr(nz, _dp), 1 if force_staged else (2 if direct else (3 if no_tconv else 0)),
                                     _ptr(eq, _dp), _ptr(dec, _i32p), _ptr(be, _i64p), _ptr(se, _i64p))
        self._check(rc)
        return eq, dec, be, se

    def ber_draws(self, s, L, seed, variant, frame_ids):
        ids = np.ascontiguousarray(frame_ids, dtype=np.int64)
        F = ids.size
        si = np.empty((F, s.S, s.N), dtype=np.int32)
        nz = np.empty((F, s.noise_len(L)), dtype=np.complex128)
        rc = load().wofdm_ber_draws(self._h, C.byref(s), L, int(seed), int(variant), _ptr(ids, _i64p), F,
                                    _ptr(si, _i32p), _ptr(nz, _dp))
        self._check(rc)
        return si, nz

    # ---- interference ----
    def interf_power(self, s, win_tx, win_rx, chan, mode=0, scalar=False):
        wt, wr, chf, L, Cn = self._win_chan(s, win_tx, win_rx, chan)
        if scalar:
            P = np.empty(Cn)
            rc = load().wofdm_interf_power_scalar(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp),
                                                  L, Cn, int(mode), _ptr(P, _dp))
        else:
            P = np.empty((Cn, s.N))
            rc = load().wofdm_interf_power(self._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp),
                                           L, Cn, int(mode), _ptr(P, _dp))
        self._check(rc)
        return P


    def interf_last_timing(self):
        """dict(total_ms, band_ms, gemm_ms, k_slice0, k_isi) of the last interf_power call (wofdm_interf_last_timing)."""
        t, b, g = C.c_double(), C.c_double(), C.c_double()
        k0, ki = C.c_int(), C.c_int()
        self._check(load().wofdm_interf_last_timing(self._h, C.byref(t), C.byref(b), C.byref(g), C.byref(k0), C.byref(ki)))
        return dict(total_ms=t.value, band_ms=b.value, gemm_ms=g.value, k_slice0=k0.value, k_isi=ki.value)

    def window_hessian(self, s, chan):
        """Hessian of the interference power in the reduced window variables (wofdm_window_hessian) for ONE impulse
        response chan (L,) -> (n_var, n_var), n_var = (tail_rx/2+1)*(tail_tx+1), index a*(tail_tx+1)+b."""
        ch = _cplx(np.ravel(chan))
        n_var = (s.tail_rx // 2 + 1) * (s.tail_tx + 1)
        H = np.empty((n_var, n_var))
        nv = C.c_int(0)
        rc = load().wofdm_window_hessian(self._h, C.byref(s), _ptr(ch, _dp), ch.size, _ptr(H, _dp), C.byref(nv))
        self._check(rc)
        assert nv.value == n_var
        return H

    def window_hessian_parts(self, s, chan, basis_tx, basis_rx):
        """The ICI and ISI parts of the quadratic form for arbitrary basis windows (wofdm_window_hessian_parts):
        basis_tx (n_tb, n_tx), basis_rx (n_rb, N + tail_rx) -> (H_ici, H_isi), each (n_var, n_var), u = a*n_tb + b."""
        ch = _cplx(np.ravel(chan))
        bt = np.ascontiguousarray(np.atleast_2d(basis_tx), dtype=np.float64)
        br = np.ascontiguousarray(np.atleast_2d(basis_rx), dtype=np.float64)
        if bt.shape[1] != s.n_tx or br.shape[1] != s.N + s.tail_rx:
            raise WofdmError(EINVAL, f"basis windows must have {s.n_tx} (Tx) and {s.N + s.tail_rx} (Rx) samples")
        n_var = bt.shape[0] * br.shape[0]
        Hc, Hs = np.empty((n_var, n_var)), np.empty((n_var, n_var))
        rc = load().wofdm_window_hessian_parts(self._h, C.byref(s), _ptr(ch, _dp), ch.size, _ptr(bt, _dp), bt.shape[0],
                                               _ptr(br, _dp), br.shape[0], _ptr(Hc, _dp), _ptr(Hs, _dp))
        self._check(rc)
        return Hc, Hs

    @staticmethod
    def _chan_set(chans):
        """(L, C) channel set (a 1-D array is one channel) -> contiguous (C, L) complex128 == L x C column-major, L, C"""
        ch = np.asarray(chans)
        if ch.ndim == 1:
            ch = ch[:, None]
        if ch.ndim != 2:
            raise WofdmError(EINVAL, "channel set must be an (L, C) array")
        return _cplx(ch.T), ch.shape[0], ch.shape[1]

    def window_hessian_set(self, s, chans):
        """Mean over the channel set chans (L, C) of window_hessian (wofdm_window_hessian_set): the quadratic form of the
        expected interference power over the set, (n_var, n_var), same variable order as window_hessian."""
        chf, L, Cn = self._chan_set(chans)
        n_var = (s.tail_rx // 2 + 1) * (s.tail_tx + 1)
        H = np.empty((n_var, n_var))
        nv = C.c_int(0)
        rc = load().wofdm_window_hessian_set(self._h, C.byref(s), _ptr(chf, _dp), L, Cn, _ptr(H, _dp), C.byref(nv))
        self._check(rc)
        assert nv.value == n_var
        return H

    def window_hessian_parts_set(self, s, chans, basis_tx, basis_rx):
        """Mean over the channel set chans (L, C) of window_hessian_parts (wofdm_window_hessian_parts_set) -> (H_ici, H_isi)."""
        chf, L, Cn = self._chan_set(chans)
        bt = np.ascontiguousarray(np.atleast_2d(basis_tx), dtype=np.float64)
        br = np.ascontiguousarray(np.atleast_2d(basis_rx), dtype=np.float64)
        if bt.shape[1] != s.n_tx or br.shape[1] != s.N + s.tail_rx:
            raise WofdmError(EINVAL, f"basis windows must have {s.n_tx} (Tx) and {s.N + s.tail_rx} (Rx) samples")
        n_var = bt.shape[0] * br.shape[0]
        Hc, Hs = np.empty((n_var, n_var)), np.empty((n_var, n_var))
        rc = load().wofdm_window_hessian_parts_set(self._h, C.byref(s), _ptr(chf, _dp), L, Cn, _ptr(bt, _dp), bt.shape[0],
                                                   _ptr(br, _dp), br.shape[0], _ptr(Hc, _dp), _ptr(Hs, _dp))
        self._check(rc)
        return Hc, Hs

    def window_hessian_last_timing(self):
        """dict(device_ms, factor_ms, passes) of the last window_hessian* call (wofdm_window_hessian_last_timing)."""
        t, f, n = C.c_double(), C.c_double(), C.c_int()
        self._check(load().wofdm_window_hessian_last_timing(self._h, C.byref(t), C.byref(f), C.byref(n)))
        return dict(device_ms=t.value, factor_ms=f.value, passes=n.value)

    def gen_channels(self, standard, L, doppler_freq, sampling_rate, frame_duration, no_frames=1, n_sets=1, seed=0,
                     phases=None):
        """ITU-R channels with GMEDS_1 fading (wofdm_gen_channels) -> (L, n_sets*no_frames) complex128.
        phases: None (on-device Philox draws) or (n_sets, n_paths, 21, 2) standard-normal draws."""
        prof = load().wofdm_channel_profile(str(standard).encode())
        if prof < 0:
            raise WofdmError(EINVAL, f"unknown ITU-R channel profile {standard!r}")
        ph = None
        if phases is not None:
            ph = _f64(np.ascontiguousarray(phases, dtype=np.float64).ravel())
            if ph.size % (int(n_sets) * 21 * 2):
                raise WofdmError(EINVAL, "phases must have shape (n_sets, n_paths, 21, 2)")
        out = np.empty((int(n_sets) * int(no_frames), int(L)), dtype=np.complex128)
        rc = load().wofdm_gen_channels(self._h, prof, int(L), float(doppler_freq), float(sampling_rate),
                                       float(frame_duration), int(no_frames), int(n_sets), int(seed),
                                       _ptr(ph, _dp) if ph is not None else None, _ptr(out, _dp))
        self._check(rc)
        return out.T


def _roll_offs(roll_offs, n_var):
    """a scalar roll-off for every pair, or n_var of them -> contiguous int32 (n_var,)"""
    ro = np.atleast_1d(np.asarray(roll_offs))
    if ro.ndim != 1 or ro.size not in (1, n_var) or not np.all(ro == np.round(ro)):
        raise WofdmError(EINVAL, f"roll_offs must be one integer or {n_var} of them (one per window pair)")
    return np.ascontiguousarray(np.broadcast_to(ro, (n_var,)), dtype=np.int32)


def _resolve(s, n, Cn, by_subcarrier, by_channel):
    """WOFDM_BY_* flags and the counter shape (n_snr, Cr, Nr) they give, (n_snr,) without them."""
    resolve = (WOFDM_BY_SUBCARRIER if by_subcarrier else 0) | (WOFDM_BY_CHANNEL if by_channel else 0)
    return resolve, ((n, Cn if by_channel else 1, s.N if by_subcarrier else 1) if resolve else (n,))


def _target(target_bit_errors, target_symbol_errors):
    """(target_kind, target) of the adaptive calls, from exactly one of the two targets."""
    if (target_bit_errors is None) == (target_symbol_errors is None):
        raise WofdmError(EINVAL, "give exactly one of target_bit_errors / target_symbol_errors")
    return ((WOFDM_TARGET_BIT_ERRORS, target_bit_errors) if target_bit_errors is not None
            else (WOFDM_TARGET_SYMBOL_ERRORS, target_symbol_errors))


def reduce_trampoline(fn, shape=None):
    """A wofdm_reduce_fn calling fn(counts) on the int64 counts of a round (a numpy view, reshaped to `shape`).  fn returns
    the summed counts (copied back) or None (it summed in place).  An exception is kept in `.error` and reported to the
    library as a non-zero return, which fails the call: ctypes would otherwise print and swallow it, and the run would go
    on with unsummed counts.  Keep the returned object alive for the duration of the call."""
    def tramp(ptr, n, user):
        try:
            a = np.ctypeslib.as_array(ptr, shape=(int(n),))
            v = a.reshape(shape) if shape is not None else a
            r = fn(v)
            if r is not None:
                r = np.asarray(r.cpu() if hasattr(r, "cpu") else r, dtype=np.int64)
                if r.size != a.size:
                    raise ValueError(f"reduce returned {r.size} counts, expected {a.size}")
                a[:] = r.reshape(-1)
            return 0
        except BaseException as e:       # noqa: BLE001 -- reported through the return value
            cb.error = e
            return 1
    cb = REDUCE_FN(tramp)
    cb.error = None
    return cb


class BerPlan:
    """Device-resident inputs of one (system, windows, channel set, SNR grid); asynchronous launches."""

    def __init__(self, handle, s, win_tx, win_rx, chan, snr_db, multi=False):
        self.handle, self.sys = handle, s
        snr = _f64(np.ravel(snr_db))
        self._p = C.c_void_p()
        if multi:
            wt, wr = handle._win_multi(s, win_tx, win_rx)
            _, _, chf, L, Cn = handle._win_chan(s, wt[0], wr[0], chan)
            self.n_var = wt.shape[0]
            rc = load().wofdm_ber_plan_create_multi(handle._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), self.n_var, _ptr(chf, _dp),
                                                    L, Cn, _ptr(snr, _dp), snr.size, C.byref(self._p))
        else:
            wt, wr, chf, L, Cn = handle._win_chan(s, win_tx, win_rx, chan)
            self.n_var = 1
            rc = load().wofdm_ber_plan_create(handle._h, C.byref(s), _ptr(wt, _dp), _ptr(wr, _dp), _ptr(chf, _dp), L, Cn,
                                              _ptr(snr, _dp), snr.size, C.byref(self._p))
        self.n_snr, self.L, self.C = snr.size, L, Cn
        handle._check(rc)
        handle._plans.add(self)

    @property
    def kernel(self):
        return load().wofdm_ber_plan_kernel(self._p).decode()

    def launch(self, ensemble, seed=0, variant=0, shard=(0, 1), slot=0, stream=None):
        """Asynchronous.  Returns the device address of the int64[n_snr][2] counters."""
        d = C.c_void_p()
        rc = load().wofdm_ber_plan_launch(self._p, slot, int(ensemble), int(seed), int(variant), int(shard[0]),
                                          int(shard[1]), C.c_void_p(stream) if stream else None, C.byref(d))
        self.handle._check(rc)
        return d.value

    @property
    def fused(self):
        """True if one launch evaluates all window pairs of the plan."""
        f = C.c_int(0)
        load().wofdm_ber_plan_variants(self._p, C.byref(f))
        return bool(f.value)

    def read(self):
        """(bit_err, sym_err): (n_snr,) each, or (n_var, n_snr) for a multi-variant plan."""
        shape = (self.n_var, self.n_snr) if self.n_var > 1 else (self.n_snr,)
        be, se = np.zeros(shape, dtype=np.int64), np.zeros(shape, dtype=np.int64)
        self.handle._check(load().wofdm_ber_plan_read(self._p, _ptr(be, _i64p), _ptr(se, _i64p)))
        return be, se

    def totals(self, ensemble, shard=(0, 1)):
        """(bit_tot, sym_tot) per SNR point for frames f = shard[0] mod shard[1]."""
        from .sharding import totals
        return totals(self.n_snr, self.C, ensemble, self.sys.n_active, self.sys.S, self.sys.bits, shard)

    def close(self):
        if getattr(self, "_p", None):
            load().wofdm_ber_plan_destroy(self._p)
            self._p = None

    __del__ = close
