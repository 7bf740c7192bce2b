"""Host-side mirror of the reference's Hessian builders, backed by libwofdm.so (SURVEY.md section 8f-2).

``OptimizerTx(system, dft_len, cp_len, tail_len)``, ``OptimizerRx(...)`` and
``OptimizerTxRx(system, dft_len, cp_len, tail_tx_len, tail_rx_len)`` keep the constructors and the two methods the
reference's ``optimization_fun`` calls before the QP / trust-region solve
(python/optimization_tools/optimizers.py:180-257, 330-410, 735-833):

    chann = opt.calculate_chann_matrices(channel_ir)      # here: just the impulse response (the device builds H_m)
    H = opt.gen_hessian(chann)                            # one device call instead of the O(n^2 N^2) loops
    H = opt.gen_hessian_expected(channels)                # or: the expected interference over the whole (L, C) set

The solvers themselves (quadratic_solver, scipy trust-constr) are the reference's and stay on the CPU: they are
sequential 9- to 54-variable problems (SURVEY section 2, out of scope).  No CPU fallback for the Hessian."""
from __future__ import annotations

import numpy as np

from . import capi, ofdm_utils


class _Base:
    def __init__(self, name, dft_len, cp_len, tail_tx, tail_rx, handle=None):
        self.name, self.dft_len, self.cp_len = name, dft_len, cp_len
        self._sys = capi.params_from_name(name, dft_len, cp_len, tail_tx, tail_rx)     # raises on unknown names
        self.cs_len, self.rm_len, self.shift_len = self._sys.cs, self._sys.rm, self._sys.shift
        self._h = handle

    def calculate_chann_matrices(self, channel_ir):
        return np.asarray(channel_ir, dtype=np.complex128).ravel()

    def gen_hessian(self, channel_tensor):
        h = self._h or ofdm_utils.default_handle()
        return h.window_hessian(self._sys, channel_tensor)

    def gen_hessian_expected(self, channels):
        """Hessian of the interference power averaged over every realisation of the stored set: channels (L, C) as the
        reference stores them (channels/<standard>.npy), instead of gen_hessian on their mean impulse response.  The
        mean of C zero-mean Rayleigh channels is one random channel of covariance R / C, not a typical one."""
        h = self._h or ofdm_utils.default_handle()
        return h.window_hessian_set(self._sys, channels)


class OptimizerTx(_Base):
    def __init__(self, system_design, dft_len, cp_len, tail_len, handle=None):
        if system_design not in ("wtx", "CPwtx"):
            raise ValueError(f"OptimizerTx handles wtx and CPwtx, not {system_design!r}")
        super().__init__(system_design, dft_len, cp_len, tail_len, 0, handle)
        self.tail_len = tail_len


class OptimizerRx(_Base):
    def __init__(self, system_design, dft_len, cp_len, tail_len, handle=None):
        if system_design not in ("wrx", "CPwrx"):
            raise ValueError(f"OptimizerRx handles wrx and CPwrx, not {system_design!r}")
        super().__init__(system_design, dft_len, cp_len, 0, tail_len, handle)
        self.tail_len = tail_len


class OptimizerTxRx(_Base):
    def __init__(self, system_design, dft_len, cp_len, tail_tx_len, tail_rx_len, handle=None):
        if system_design not in ("WOLA", "CPW"):
            raise ValueError(f"OptimizerTxRx handles WOLA and CPW, not {system_design!r}")
        super().__init__(system_design, dft_len, cp_len, tail_tx_len, tail_rx_len, handle)
        self.tail_tx_len, self.tail_rx_len = tail_tx_len, tail_rx_len
