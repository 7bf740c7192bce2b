"""CPU port of the reference's Monte-Carlo loop for TIMING  --  TEST/BENCH INFRASTRUCTURE ONLY.

``bench.py``'s ``cpu_baseline`` leg and ``bench.py --impl reference`` time this module on the GPU
box's host cores (the reference itself is not part of this repository).  It
restates python/ofdm_utils/wofdm_simulation.py:171-240 with the reference's own cost profile:
numba-jitted, single-threaded per task, dense ``tx_mat @ X`` / ``rx_mat @ frame`` products
(:187, :221), ``np.convolve`` (:206), exact-SNR AWGN (:135-138), and the 16-way ``argmin |sym - x|``
decision per sample (:159-164).  Tasks fan out over processes as the reference's driver does
(python/wofdm_optimization.py:127-131, ``Pool(cpu_count())``).

The product path never imports this file.  Correctness of the port is pinned in
tests/test_oracle_golden.py::test_cpu_port_statistics against the numpy oracle.
"""
from __future__ import annotations

import os
import time

import numpy as np
from numba import njit

from . import wofdm_oracle as O


@njit(cache=True, fastmath=True)
def _mc_dense(tx_mat, rx_mat, n_sym, channels, ensemble, snr_arr, tail_tx, points, seed):
    """Symbol-error counts per SNR point; one window pair (the reference runs two per frame)."""
    np.random.seed(seed)
    n_sub = tx_mat.shape[1]
    n_tx = tx_mat.shape[0]
    stride = rx_mat.shape[1]
    n_pts = points.shape[0]
    L = channels.shape[0]
    keep = n_sym * stride
    errs = np.zeros(snr_arr.shape[0], dtype=np.int64)
    X = np.empty((n_sub, n_sym), dtype=np.complex128)
    for si in range(snr_arr.shape[0]):
        gain = 10.0 ** (-0.1 * snr_arr[si])
        for c in range(channels.shape[1]):
            h = channels[:, c].copy()
            for _e in range(ensemble):
                for k in range(n_sub):
                    for s in range(n_sym):
                        X[k, s] = points[np.random.randint(0, n_pts)]
                blocks = np.ascontiguousarray((tx_mat @ X).T)            # (S, n_tx)        :187
                u = np.zeros(tail_tx + keep, dtype=np.complex128)
                for s in range(n_sym):                                   # overlap-add      :190-203
                    u[s * stride: s * stride + n_tx] += blocks[s]
                r = np.convolve(h, u)[:keep]                             #                  :206-209
                n = np.random.randn(keep) + 1j * np.random.randn(keep)   #                  :136
                px = np.sum(r.real * r.real + r.imag * r.imag)
                pn = np.sum(n.real * n.real + n.imag * n.imag)
                y = r + np.sqrt(px * gain / pn) * n                      #                  :138-140
                Y = rx_mat @ np.ascontiguousarray(y.reshape(n_sym, stride).T)   # (N, S)   :217-221
                for k in range(n_sub):
                    hest = Y[k, 0] / X[k, 0]                             #                  :223
                    for s in range(1, n_sym):
                        v = Y[k, s] / hest                               #                  :231
                        best = 0
                        dmin = np.abs(points[0] - v)
                        for q in range(1, n_pts):                        # argmin           :163
                            d = np.abs(points[q] - v)
                            if d < dmin:
                                dmin = d
                                best = q
                        if points[best] != X[k, s]:                      #                  :235
                            errs[si] += 1
    return errs


def build_task(name, N, cp, tail_tx, tail_rx, S, bits, channels, ensemble, snr_arr, seed, v_tx=None, v_rx=None):
    p = O.system_params(name, N, cp, tail_tx, tail_rx, S=S, bits=bits)
    vt = O.rc_window_tx(p) if v_tx is None else v_tx
    vr = O.rc_window_rx(p) if v_rx is None else v_rx
    return dict(tx_mat=O.tx_matrix(p, vt), rx_mat=O.rx_matrix(p, vr), S=S, channels=np.ascontiguousarray(channels),
                ensemble=int(ensemble), snr=np.ascontiguousarray(snr_arr, dtype=np.float64), tail_tx=tail_tx,
                points=O.qam_points(bits, 0), seed=int(seed), N=N)


def run_task(t):
    return _mc_dense(t["tx_mat"], t["rx_mat"], t["S"], t["channels"], t["ensemble"], t["snr"], t["tail_tx"],
                     t["points"], t["seed"])


_LIMIT = None


def _warm(_=None):
    """JIT-compile (or load the cache) and pin BLAS to one thread per process: the reference's fan-out
    is over processes (wofdm_optimization.py:127-131).  scipy's OpenBLAS, which numba's ``@`` calls, is
    only loaded by the first jitted call, so the limit is applied after it."""
    global _LIMIT
    p = O.system_params("wtx", 16, 4, 2, 0, S=3)
    t = dict(tx_mat=O.tx_matrix(p, O.rc_window_tx(p)), rx_mat=O.rx_matrix(p, O.rc_window_rx(p)), S=3,
             channels=np.ones((2, 1), dtype=np.complex128), ensemble=1, snr=np.array([10.0]), tail_tx=2,
             points=O.qam_points(4, 0), seed=0, N=16)
    run_task(t)
    try:
        from threadpoolctl import threadpool_limits
        _LIMIT = threadpool_limits(limits=1)
    except Exception:   # pragma: no cover
        pass
    return os.getpid()


def timed_throughput(tasks, workers):
    """OFDM symbols/s over `tasks` with `workers` processes; JIT compilation excluded."""
    syms = sum(len(t["snr"]) * t["channels"].shape[1] * t["ensemble"] * t["S"] for t in tasks)
    if workers <= 1:
        _warm()
        t0 = time.perf_counter()
        out = [run_task(t) for t in tasks]
        dt = time.perf_counter() - t0
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(workers, initializer=_warm) as pool:
            pool.map(_warm, range(workers))          # every worker is up and JIT-warm before the clock starts
            t0 = time.perf_counter()
            out = pool.map(run_task, tasks, chunksize=1)
            dt = time.perf_counter() - t0
    return syms / dt, dt, syms, out
