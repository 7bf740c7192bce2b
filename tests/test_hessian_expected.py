"""Window Hessian averaged over a channel set (wofdm_window_hessian_set / _parts_set): the quadratic form of the EXPECTED
interference power over every realisation, instead of the Hessian of the mean impulse response.

The device path rests on one identity: H(h) is a linear function of h h^H, so
    (1/C) sum_c H(h_c) = sum_j H(g_j)   for any factor G = [g_1 .. g_r] of R = (1/C) sum_c h_c h_c^H.
CPU tests check that identity on the oracle, for an eigenvector factor and for the pivoted Cholesky factor the library
uses (restated here in numpy); GPU tests check the device against the plain mean of the single-channel oracle."""
import ctypes
import os

import numpy as np
import pytest

from oracle import hessian_set as HS
from oracle import wofdm_oracle as O

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hessian.npz"))
SYSTEMS = ("wtx", "CPwtx", "wrx", "CPwrx", "WOLA", "CPW")
FACTOR_TOL = 1e-14          # the library's kSetFactorTol (csrc/interf.cu)


def tails(name, ttx, trx):
    return (ttx if name in ("wtx", "CPwtx", "WOLA", "CPW") else 0, trx if name in ("wrx", "CPwrx", "WOLA", "CPW") else 0)


def covariance(chans):
    return chans @ chans.conj().T / chans.shape[1]


def eig_factor(chans):
    lam, V = np.linalg.eigh(covariance(chans))
    keep = lam > 0
    return V[:, keep] * np.sqrt(lam[keep])


def pivoted_cholesky(R, tol=FACTOR_TOL):
    """The library's factorisation (channel_set_factor, csrc/interf.cu): columns g_k with R ~= sum_k g_k g_k^H, pivot =
    the largest remaining diagonal entry, stop when it is at most tol times the largest diagonal entry of R."""
    L = R.shape[0]
    d = R.diagonal().real.copy()
    dmax = d.max()
    used = np.zeros(L, dtype=bool)
    cols = []
    for _ in range(L):
        p = int(np.argmax(np.where(used, -np.inf, d)))
        if not d[p] > tol * dmax:
            break
        s = np.sqrt(d[p])
        used[p] = True
        g = np.zeros(L, dtype=np.complex128)
        rest = ~used
        acc = R[:, p].copy()
        for gj in cols:
            acc -= gj * np.conj(gj[p])
        g[rest] = acc[rest] / s
        d[rest] -= np.abs(g[rest]) ** 2
        g[p] = s
        cols.append(g)
    return np.stack(cols, axis=1) if cols else np.zeros((L, 1), dtype=np.complex128)


def hessian_of_factor(p, F):
    return sum(O.window_hessian(p, F[:, j]) for j in range(F.shape[1]))


def rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


# ---- CPU: the identity the device path relies on ---------------------------------------------------------------------

@pytest.mark.parametrize("name", ["WOLA", "CPwrx"])
def test_factor_identity(name):
    a, b = tails(name, 2, 2)
    p = O.system_params(name, 64, 8, a, b)
    chans = O.synth_channels(40, 9, seed=1)
    want = HS.window_hessian_set(p, chans)
    F_eig = eig_factor(chans)
    F_chol = pivoted_cholesky(covariance(chans))
    assert F_chol.shape[1] <= 9
    assert np.abs(F_chol @ F_chol.conj().T - covariance(chans)).max() <= 1e-14 * np.abs(covariance(chans)).max()
    assert rel(hessian_of_factor(p, F_eig), want) <= 1e-12
    assert rel(hessian_of_factor(p, F_chol), want) <= 1e-12


def test_rank_deficient_sets():
    """Three channels repeated ten times (C = 30 > L: factored, rank 3) and a set smaller than L (C = 4: the channels
    themselves or their factor): the same Hessian either way."""
    p = O.system_params("WOLA", 64, 8, 2, 2)
    rng = np.random.default_rng(7)
    base = (rng.standard_normal((9, 3)) + 1j * rng.standard_normal((9, 3))) * np.exp(-np.arange(9) / 3.0)[:, None]
    rep = np.repeat(base, 10, axis=1)
    F = pivoted_cholesky(covariance(rep))
    assert F.shape[1] == 3
    direct = HS.window_hessian_set(p, base)                 # the mean over the repeated set = the mean over the three
    assert rel(hessian_of_factor(p, F), direct) <= 1e-12
    small = O.synth_channels(4, 9, seed=3)
    F4 = pivoted_cholesky(covariance(small))
    assert F4.shape[1] == 4
    want = HS.window_hessian_set(p, small)
    assert rel(hessian_of_factor(p, F4), want) <= 1e-12
    assert rel(sum(O.window_hessian(p, small[:, c]) for c in range(4)) / 4, want) <= 1e-15


@pytest.mark.parametrize("name", ["WOLA", "wtx", "wrx"])
def test_quadratic_form_is_mean_interference(name):
    """0.5 x^T H_set x = the mean over the set of the interference power of the expanded windows (ISI slices summed
    before squaring: interf_power_matlab)."""
    a, b = tails(name, 2, 2)
    p = O.system_params(name, 64, 8, a, b)
    chans = O.synth_channels(12, 9, seed=5)
    H = HS.window_hessian_set(p, chans)
    rng = np.random.default_rng(2)
    xt = np.concatenate([[1.0], rng.uniform(0, 1, a)])
    xr = np.concatenate([[1.0], rng.uniform(0.5, 1, b // 2)])
    x = np.outer(xr, xt).ravel()
    vt, vr = O.expand_window_tx(xt, p), O.expand_window_rx(xr, p)
    want = np.mean([O.interf_power_matlab(p, vt, vr, chans[:, c]) for c in range(chans.shape[1])])
    assert abs(0.5 * x @ H @ x - want) <= 1e-9 * want


def test_quad_objective_expected_oracle_is_mean_of_quad_objective():
    p = O.system_params("WOLA", 16, 4, 2, 2)
    vt, vr, _, _ = O.perturbed_windows(p, seed=3)
    chans = O.synth_channels(3, 5, seed=2)
    for side, fixed in (("tx", vr), ("rx", vt)):
        want = np.mean([O.quad_objective_matlab(p, side, fixed, chans[:, c], 0.3) for c in range(3)], axis=0)
        assert rel(HS.quad_objective_expected(p, side, fixed, chans, 0.3), want) <= 1e-12


# ---- GPU: the device path against the oracle --------------------------------------------------------------------------

def _sys(W, name, N, cp, a, b):
    return W.params_from_name(name, N, cp, a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SYSTEMS)
def test_device_set_matches_oracle_n64(name):
    """Golden system (N = 64, cp 10, tails 4 / 6, 9 taps): C = 5 <= L (the channels themselves) against the plain mean;
    C = 250 (factored) against the oracle evaluated on an eigenvector factor of the set's covariance (the identity the CPU
    tests pin), and for WOLA against the plain mean of all 250 single-channel Hessians as well."""
    import wofdm_b200 as W
    a, b = tails(name, int(G["tail_tx"]), int(G["tail_rx"]))
    N, cp = int(G["N"]), int(G["cp"])
    p = O.system_params(name, N, cp, a, b)
    s = _sys(W, name, N, cp, a, b)
    small = O.synth_channels(5, 9, seed=11)
    big = O.synth_channels(250, 9, seed=1)
    with W.Handle([0]) as h:
        Hd = h.window_hessian_set(s, small)
        assert h.window_hessian_last_timing()["passes"] == 5
        want = HS.window_hessian_set(p, small)
        assert np.abs(Hd - want).max() <= 1e-9 * np.abs(want).max()
        Hd = h.window_hessian_set(s, big)
        assert h.window_hessian_last_timing()["passes"] <= 9
        want = hessian_of_factor(p, eig_factor(big))
        assert np.abs(Hd - want).max() <= 1e-9 * np.abs(want).max()
        if name == "WOLA":
            want = HS.window_hessian_set(p, big)
            assert np.abs(Hd - want).max() <= 1e-9 * np.abs(want).max()
        assert np.array_equal(Hd, Hd.T)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["WOLA", "CPW"])
def test_device_set_matches_oracle_n256(name):
    """settingsData sizes: N = 256, tails 8 / 10, 21 taps; C = 3 <= L and C = 250 (VehA: rank 6, six passes)."""
    import wofdm_b200 as W
    p = O.system_params(name, 256, 16, 8, 10)
    s = _sys(W, name, 256, 16, 8, 10)
    small = O.synth_channels(3, 21, seed=12)
    big = O.synth_channels(250, 21, seed=1)
    with W.Handle([0]) as h:
        Hd = h.window_hessian_set(s, small)
        want = HS.window_hessian_set(p, small)
        assert np.abs(Hd - want).max() <= 1e-9 * np.abs(want).max()
        Hd = h.window_hessian_set(s, big)
        t = h.window_hessian_last_timing()
        assert t["passes"] <= 21 and t["device_ms"] > 0
        want = hessian_of_factor(p, eig_factor(big))
        assert np.abs(Hd - want).max() <= 1e-9 * np.abs(want).max()
        print(f"{name}: C = 250 in {t['passes']} passes, device {t['device_ms']:.2f} ms, factor {t['factor_ms']:.3f} ms")


@pytest.mark.gpu
def test_single_channel_set_is_bitwise_window_hessian():
    import wofdm_b200 as W
    from wofdm_b200 import optimizers as OPT
    hch = O.synth_channels(1, 21, seed=4)
    with W.Handle([0]) as h:
        for name, a, b in (("WOLA", 8, 10), ("wtx", 8, 0), ("CPwrx", 0, 10)):
            s = _sys(W, name, 256, 16, a, b)
            assert np.array_equal(h.window_hessian_set(s, hch), h.window_hessian(s, hch[:, 0]))
        p = O.system_params("WOLA", 64, 8, 2, 2)
        s = _sys(W, "WOLA", 64, 8, 2, 2)
        bt, br = O.window_basis(p)
        ch = O.synth_channels(1, 9, seed=6)
        Hc1, Hs1 = h.window_hessian_parts(s, ch[:, 0], bt, br)
        Hc2, Hs2 = h.window_hessian_parts_set(s, ch, bt, br)
        assert np.array_equal(Hc1, Hc2) and np.array_equal(Hs1, Hs2)
        opt = OPT.OptimizerTxRx("WOLA", 64, 8, 2, 2, handle=h)
        assert np.array_equal(opt.gen_hessian_expected(ch), opt.gen_hessian(opt.calculate_chann_matrices(ch[:, 0])))


@pytest.mark.gpu
@pytest.mark.parametrize("C", [5, 30])
def test_identical_channels_give_the_single_channel_hessian(C):
    """C copies of one channel: C <= L runs C passes, C > L factors a rank-1 covariance into one pass."""
    import wofdm_b200 as W
    hch = O.synth_channels(1, 21, seed=8)[:, 0]
    with W.Handle([0]) as h:
        s = _sys(W, "CPW", 256, 16, 8, 10)
        Hs = h.window_hessian_set(s, np.repeat(hch[:, None], C, axis=1))
        assert h.window_hessian_last_timing()["passes"] == (C if C <= 21 else 1)
        H1 = h.window_hessian(s, hch)
        assert np.abs(Hs - H1).max() <= 1e-12 * np.abs(H1).max()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 30])
def test_parts_and_quad_objective_expected_match_oracle(C):
    import wofdm_b200 as W
    from wofdm_b200 import ofdm_utils as U
    from wofdm_b200 import optimizers as OPT
    N, cp, ttx, trx = 64, 8, 2, 2
    p = O.system_params("WOLA", N, cp, ttx, trx)
    s = _sys(W, "WOLA", N, cp, ttx, trx)
    vt, vr, _, _ = O.perturbed_windows(p, seed=9)
    chans = O.synth_channels(C, 9, seed=13)
    with W.Handle([0]) as h:
        bt, br = O.window_basis(p)
        Hc, Hs = h.window_hessian_parts_set(s, chans, bt, br)
        wc, ws = HS.window_hessian_parts_set(p, chans, bt, br)
        assert np.abs(Hc - wc).max() <= 1e-9 * np.abs(wc).max()
        assert np.abs(Hs - ws).max() <= 1e-9 * np.abs(ws).max()
        HTx = U.quad_objective_tx_expected(np.diag(vr), N, trx, cp, "WOLA", ttx, chans.T, 0.5, handle=h)
        want = HS.quad_objective_expected(p, "tx", vr, chans, 0.5)
        assert HTx.shape == (p.n_tx, p.n_tx)
        assert np.abs(HTx - want).max() <= 1e-9 * np.abs(want).max()
        HRx = U.quad_objective_rx_expected(vt, N, trx, cp, "WOLA", ttx, chans.T, 0.25, handle=h)
        want = HS.quad_objective_expected(p, "rx", vt, chans, 0.25)
        assert np.abs(HRx - want).max() <= 1e-9 * np.abs(want).max()
        opt = OPT.OptimizerTxRx("WOLA", N, cp, ttx, trx, handle=h)
        H = opt.gen_hessian_expected(chans)
        want = HS.window_hessian_set(p, chans)
        assert np.abs(H - want).max() <= 1e-9 * np.abs(want).max()


@pytest.mark.gpu
def test_error_codes():
    import wofdm_b200 as W
    from wofdm_b200 import capi
    lib = capi.load()
    dp = ctypes.POINTER(ctypes.c_double)
    chans = np.ascontiguousarray(O.synth_channels(4, 9, seed=1).T)
    H = np.empty((9 * 9,))
    p = O.system_params("WOLA", 64, 8, 2, 2)
    bt, br = (np.ascontiguousarray(x) for x in O.window_basis(p))
    Hc, Hs = np.empty(81), np.empty(81)
    with W.Handle([0]) as h:
        s = _sys(W, "WOLA", 64, 8, 2, 2)

        def hs(sys_, ch, L, C, out):
            return lib.wofdm_window_hessian_set(h._h, ctypes.byref(sys_), ch, L, C, out, None)

        def ps(sys_, ch, L, C, b_tx, b_rx):
            return lib.wofdm_window_hessian_parts_set(h._h, ctypes.byref(sys_), ch, L, C, b_tx, 3, b_rx, 2,
                                                      Hc.ctypes.data_as(dp), Hs.ctypes.data_as(dp))
        cp_, hp = chans.ctypes.data_as(dp), H.ctypes.data_as(dp)
        btp, brp = bt.ctypes.data_as(dp), br.ctypes.data_as(dp)
        assert hs(s, cp_, 9, 4, hp) == capi.OK
        assert hs(s, cp_, 9, 0, hp) == capi.EINVAL
        assert b"C must be" in lib.wofdm_last_error(h._h)
        assert hs(s, None, 9, 4, hp) == capi.EINVAL
        assert hs(s, cp_, 9, 4, None) == capi.EINVAL
        bad = chans.copy()
        bad[2, 3] = np.nan
        assert hs(s, bad.ctypes.data_as(dp), 9, 4, hp) == capi.EINVAL
        assert b"non-finite" in lib.wofdm_last_error(h._h)
        bad[2, 3] = np.inf
        assert hs(s, bad.ctypes.data_as(dp), 9, 4, hp) == capi.EINVAL
        assert hs(s.copy(tail_rx=3), cp_, 9, 4, hp) == capi.EINVAL                    # validate_sys
        assert hs(s, cp_, 0, 4, hp) == capi.EINVAL                                   # L < 1
        assert hs(_sys(W, "WOLA", 32, 8, 2, 2), cp_, 9, 4, hp) == capi.EUNSUPPORTED   # N % 64
        assert ps(s, cp_, 9, 4, btp, brp) == capi.OK
        assert ps(s, cp_, 9, 0, btp, brp) == capi.EINVAL
        assert ps(s, cp_, 9, 4, None, brp) == capi.EINVAL
        assert ps(s, cp_, 9, 4, btp, None) == capi.EINVAL
        assert ps(s, bad.ctypes.data_as(dp), 9, 4, btp, brp) == capi.EINVAL
        with pytest.raises(W.WofdmError) as e:
            h.window_hessian_set(s, np.zeros((9, 0), dtype=complex))
        assert e.value.code == capi.EINVAL


@pytest.mark.gpu
def test_two_device_handle_matches_one_device():
    import wofdm_b200 as W
    n = ctypes.c_int(0)
    W.capi.load().wofdm_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs two GPUs")
    s = _sys(W, "WOLA", 256, 16, 8, 10)
    chans = O.synth_channels(250, 21, seed=2)
    with W.Handle([0]) as h1, W.Handle([0, 1]) as h2:
        H1, H2 = h1.window_hessian_set(s, chans), h2.window_hessian_set(s, chans)
    assert np.abs(H1 - H2).max() <= 1e-12 * np.abs(H1).max()
