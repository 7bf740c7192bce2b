"""PSD of the channel-mask chain's Tx streams for several windows and roll-offs on the same frames in one call
(wofdm_psd_masked_multi, Handle.psd_masked_multi, ofdm_utils.psd_sim_mc_multi).

GPU: spectrum v equals psd_masked with window v and roll_off[v] to fp64 summation order (a pair's product output does not
depend on the other pairs), under both estimators and across product batches; a NULL half is skipped; frame ranges add up;
the mirror equals psd_sim_mc per configuration; one symbol draw, one product and one PSD launch per batch whatever n_var;
the refusals leave the handle usable; a two-device handle gives the one-device spectra.
"""
import ctypes as C

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import capi, ofdm_utils as U
from oracle import wofdm_oracle as O
from test_psd_masked import chain_params, sys_of

ROLL_OFFS = [4, 10, 30, 6, 14, 20, 40, 8]


@pytest.fixture(scope="module")
def handle():
    h = W.Handle([0])
    yield h
    h.close()


def windows(p, n_var):
    """window 0: RC; window v > 0: RC perturbed by a seeded +-10 %"""
    return np.array([O.rc_window_tx(p)] + [O.perturbed_windows(p, seed=100 + v)[0] for v in range(1, n_var)])


def check_against_singles(handle, s, wt, ro, **kw):
    mm, mu = handle.psd_masked_multi(s, wt, roll_offs=ro, **kw)
    n_var = len(ro)
    assert mm.shape == mu.shape == (n_var, 8 * s.N)
    for v in range(n_var):
        sm, su = handle.psd_masked(s, wt[v], roll_off=ro[v], **kw)
        np.testing.assert_allclose(mm[v], sm, rtol=1e-12, atol=0)
        np.testing.assert_allclose(mu[v], su, rtol=1e-12, atol=0)
    if n_var > 1:
        for x in (mm, mu):
            assert all(not np.allclose(x[0], x[v], rtol=1e-6, atol=0) for v in range(1, n_var))
    return mm, mu


# (name, N, cp, tail_tx, tail_rx, guard, S, n_var, f0, frames)
SHAPES = [
    ("wtx", 128, 8, 4, 0, 32, 16, 3, 0, 6),
    ("wtx", 256, 16, 8, 0, 64, 16, 1, 5, 6),
    ("wtx", 256, 16, 8, 0, 64, 16, 2, 5, 6),
    ("wtx", 256, 16, 8, 0, 64, 16, 8, 5, 6),
    ("CPW", 256, 16, 8, 8, 64, 16, 3, 100, 4),
    ("WOLA", 512, 32, 16, 16, 128, 64, 3, 7, 3),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,cp,ttx,trx,guard,S,n_var,f0,F", SHAPES)
def test_spectra_equal_single_calls(handle, name, N, cp, ttx, trx, guard, S, n_var, f0, F):
    p = chain_params(name, N, cp, ttx, trx, guard, S)
    s = sys_of(p)
    for est in ("reference", "hann"):
        check_against_singles(handle, s, windows(p, n_var), ROLL_OFFS[:n_var], frames=F, f0=f0, seed=11, estimator=est)


@pytest.mark.gpu
def test_batches_halves_and_ranges(handle):
    """More frames than one product batch (S = 256: 512 frames per batch) against the single calls; a NULL half is skipped
    and the other one does not change; [0, a) and [a, b) weighted by their frame counts give [0, b)."""
    p = chain_params(S=256)
    s = sys_of(p)
    wt, ro = windows(p, 3), ROLL_OFFS[:3]
    a, b = 500, 1200
    for est in ("reference", "hann"):
        fm, fu = check_against_singles(handle, s, wt, ro, frames=b, seed=4, estimator=est)
        only_m, none_u = handle.psd_masked_multi(s, wt, roll_offs=ro, frames=b, seed=4, estimator=est, unmasked=False)
        none_m, only_u = handle.psd_masked_multi(s, wt, roll_offs=ro, frames=b, seed=4, estimator=est, masked=False)
        assert none_u is None and none_m is None
        np.testing.assert_allclose(only_m, fm, rtol=1e-12, atol=0)
        np.testing.assert_allclose(only_u, fu, rtol=1e-12, atol=0)
        am, au = handle.psd_masked_multi(s, wt, roll_offs=ro, frames=a, seed=4, estimator=est)
        bm, bu = handle.psd_masked_multi(s, wt, roll_offs=ro, frames=b - a, f0=a, seed=4, estimator=est)
        np.testing.assert_allclose((a * am + (b - a) * bm) / b, fm, rtol=1e-12, atol=0)
        np.testing.assert_allclose((a * au + (b - a) * bu) / b, fu, rtol=1e-12, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("n_var", [1, 2, 8])
def test_launches_per_batch_do_not_grow(handle, n_var):
    """A call one frame longer than one batch (131 072 / S frames) adds one symbol draw, one product and one PSD launch."""
    p = chain_params()
    s = sys_of(p)
    wt, ro = windows(p, n_var), ROLL_OFFS[:n_var]
    batch = 131072 // p.S
    counts = []
    for frames in (batch, batch + 1):
        before = handle.launches
        handle.psd_masked_multi(s, wt, roll_offs=ro, frames=frames, seed=2)
        counts.append(handle.launches - before)
    assert counts[1] - counts[0] == 3, counts


@pytest.mark.gpu
def test_psd_sim_mc_multi_mirror(handle):
    p = chain_params()
    wt, ro = windows(p, 3), [4, 10, 30]
    r = U.psd_sim_mc_multi(8, p.cp, p.cs, p.tail_tx, [np.diag(w) for w in wt], p.guard, p.N, p.bits, p.S, ro, seed=3,
                           handle=handle)
    assert set(r) == {"X_est_masked", "X_est", "obr_masked", "obr", "mf_band_masked", "mf_band", "f_axis"}
    for v in range(3):
        one = U.psd_sim_mc(8, p.cp, p.cs, p.tail_tx, np.diag(wt[v]), p.guard, p.N, p.bits, p.S, ro[v], seed=3, handle=handle)
        for k in ("X_est_masked", "X_est", "mf_band_masked", "mf_band"):
            np.testing.assert_allclose(r[k][v], one[k], rtol=1e-12, atol=0)
        for k in ("obr_masked", "obr"):
            assert r[k][v] == pytest.approx(one[k], rel=1e-12)
        assert np.array_equal(r["f_axis"], one["f_axis"])


def _raw(handle, s, wt, ro, n_var, n=2, m=True, u=True):
    P = 8 * s.N
    om = np.empty(P * max(n_var, 1)) if m else None
    ou = np.empty(P * max(n_var, 1)) if u else None
    w = np.ascontiguousarray(wt, dtype=np.float64)
    rop = None if ro is None else np.ascontiguousarray(ro, dtype=np.int32).ctypes.data_as(C.POINTER(C.c_int))
    return capi.load().wofdm_psd_masked_multi(handle._h, C.byref(s), w.ctypes.data_as(capi._dp), rop, n_var, 0, 0, n, 0,
                                              om.ctypes.data_as(capi._dp) if m else None,
                                              ou.ctypes.data_as(capi._dp) if u else None)


@pytest.mark.gpu
def test_rejections_leave_the_handle_usable(handle):
    p = chain_params()
    s = sys_of(p)
    wt = windows(p, 8)
    wt9 = np.vstack([wt, wt[:1]])
    E = capi.EINVAL
    cases = [
        dict(n_var=0),
        dict(wt=wt9, ro=ROLL_OFFS + [4], n_var=9),
        dict(ro=None),
        dict(ro=[4, 1000]),
        dict(ro=[0, 10]),
        dict(m=False, u=False),
    ]
    want = handle.psd_masked_multi(s, wt[:2], roll_offs=[4, 10], frames=2)
    for kw in cases:
        args = dict(wt=wt[:2], ro=[4, 10], n_var=2)
        args.update(kw)
        assert _raw(handle, s, args.pop("wt"), args.pop("ro"), args.pop("n_var"), **args) == E, kw
        again = handle.psd_masked_multi(s, wt[:2], roll_offs=[4, 10], frames=2)
        for x, y in zip(again, want):
            np.testing.assert_allclose(x, y, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_two_device_handle_matches_one_device(handle):
    n = C.c_int(0)
    assert capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("needs two GPUs")
    p = chain_params()
    s = sys_of(p)
    wt, ro = windows(p, 3), ROLL_OFFS[:3]
    one = handle.psd_masked_multi(s, wt, roll_offs=ro, frames=20, seed=6)
    with W.Handle([0, 1]) as h2:
        two = h2.psd_masked_multi(s, wt, roll_offs=ro, frames=20, seed=6)
    for x, y in zip(one, two):
        np.testing.assert_allclose(x, y, rtol=1e-12, atol=0)
