"""CPU oracle of the resolved BER counters  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``wofdm_ber_run_resolved`` counts errors per (SNR point, channel, sub-carrier).  This module turns the oracle's frames
(``wofdm_oracle.FrameResult``: ``dec_idx`` and the sent indices) into the same per-bin counts, in either constellation
convention: python natural order (0) or MATLAB Gray (1).  In both, a constellation index is the symbol's bit pattern, so
a bin's bit errors are the popcount of (sent XOR decided), as ``wofdm_oracle.bit_errors`` counts them for a whole frame.
The frame functions of ``wofdm_oracle`` are used as they are.
"""
from __future__ import annotations

import numpy as np

from .wofdm_oracle import FrameResult, SysParams, idx_to_levels, levels_to_idx


def per_bin_errors(p: SysParams, res: FrameResult, sym_idx: np.ndarray):
    """(sym_err, bit_err), each int64 (N,): errors of the frame's S-1 data symbols per FFT bin.  sym_idx: (N, S) sent
    indices in the convention of p (the frame functions' input).  Null bins of a guard band count nothing.  The sums
    over the bins are res.sym_err and res.bit_err."""
    tx = np.asarray(sym_idx, dtype=np.int64)[:, 1:]
    dec = np.asarray(res.dec_idx, dtype=np.int64)
    act = np.asarray(p.active, dtype=bool)
    diff = tx ^ dec
    sym = np.count_nonzero(diff, axis=1).astype(np.int64)
    bit = np.bitwise_count(diff.astype(np.uint64)).sum(axis=1).astype(np.int64)
    sym[~act] = 0
    bit[~act] = 0
    return sym, bit


def convert_indices(idx: np.ndarray, bits: int, src: int, dst: int) -> np.ndarray:
    """Constellation indices of convention src as indices of convention dst (the same lattice points)."""
    a, c = idx_to_levels(np.asarray(idx, dtype=np.int64), bits, src)
    return levels_to_idx(a, c, bits, dst)
