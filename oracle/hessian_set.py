"""CPU oracle of the channel-set window Hessian  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The window optimiser's quadratic form averaged over every realisation of a channel set, by definition: the plain mean of
the single-channel oracle (``wofdm_oracle.window_hessian`` and the Gram parts built from ``interf_matrices``) over the
columns of an (L, C) set.  The device path (``wofdm_window_hessian_set``) reaches the same matrix through a factor of the
sample tap covariance; this module deliberately does not.
"""
from __future__ import annotations

import numpy as np

from .wofdm_oracle import SysParams, interf_matrices, window_hessian


def window_hessian_set(p: SysParams, chans: np.ndarray) -> np.ndarray:
    """Mean over the columns of chans (L, C) of window_hessian: the quadratic form of the expected interference power
    over the channel set (the reference builds it from the mean impulse response instead)."""
    chans = np.asarray(chans)
    return np.mean([window_hessian(p, chans[:, c]) for c in range(chans.shape[1])], axis=0)


def window_hessian_parts(p: SysParams, h: np.ndarray, basis_tx: np.ndarray, basis_rx: np.ndarray):
    """(H_ici, H_isi) of one impulse response for arbitrary basis windows basis_tx (n_tb, n_tx), basis_rx (n_rb, N+tail_rx),
    variable u = a*n_tb + b: H_ici = 2 Re <offdiag A0_u, offdiag A0_u'>, H_isi = 2 Re <AS_u, AS_u'>."""
    x0, xs = [], []
    for a in range(basis_rx.shape[0]):
        for b in range(basis_tx.shape[0]):
            A = interf_matrices(p, basis_tx[b], basis_rx[a], h)
            x0.append((A[0] - np.diag(np.diag(A[0]))).ravel())
            xs.append(A[1:].sum(axis=0).ravel())
    x0, xs = np.array(x0), np.array(xs)
    return 2.0 * (x0 @ x0.conj().T).real, 2.0 * (xs @ xs.conj().T).real


def window_hessian_parts_set(p: SysParams, chans: np.ndarray, basis_tx: np.ndarray, basis_rx: np.ndarray):
    """Mean over the columns of chans (L, C) of window_hessian_parts."""
    chans = np.asarray(chans)
    parts = [window_hessian_parts(p, chans[:, c], basis_tx, basis_rx) for c in range(chans.shape[1])]
    return np.mean([q[0] for q in parts], axis=0), np.mean([q[1] for q in parts], axis=0)


def quad_objective_expected(p: SysParams, side: str, window_fixed: np.ndarray, chans: np.ndarray, alpha: float) -> np.ndarray:
    """Mean over the columns of chans (L, C) of quad_objective_matlab (matlab/window_optimization.m:596-680), through the
    parts with the full window of `side` as the variable: alpha H_ici + (1 - alpha) diag(row sums of H_isi) on the mean
    parts (the formula is linear in them)."""
    fixed = np.asarray(window_fixed, dtype=np.float64)[None, :]
    if side == "tx":
        Hc, Hs = window_hessian_parts_set(p, chans, np.eye(p.n_tx), fixed)
    else:
        Hc, Hs = window_hessian_parts_set(p, chans, fixed, np.eye(p.N + p.tail_rx))
    return alpha * Hc + (1.0 - alpha) * np.diag(Hs.sum(axis=1))
