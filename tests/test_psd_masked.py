"""PSD of the channel-mask chain's Tx streams, masked and unmasked (wofdm_psd_masked, matlab/main_channel_mask.m).

CPU: Parseval identities of both estimators, this file's masked_tx_stream against the oracle's masked chain, its product
form and the plain guard-band stream, the OBR split of the psd_sim_mc mirror, the window check of Handle.psd_masked.
GPU: the device's spectra of exported production frames against the oracle bin by bin (both estimators, N = 128 / 256 /
512, several systems, roll-offs and frame offsets); additivity over frame ranges and batches; the ensemble OBR and deep
out-of-band levels against the oracle's numpy draws; every rejection, each followed by a good call on the same handle;
the psd_sim_mc mirror's keys and shapes."""
import ctypes as C

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import capi, ofdm_utils as U
from oracle import wofdm_oracle as O


def chain_params(name="wtx", N=256, cp=16, ttx=8, trx=0, guard=64, S=16, bits=4):
    """bench.py's mask_chain shape by default: MATLAB conventions, guard band N/4"""
    return O.system_params(name, N, cp, ttx, trx, S=S, bits=bits, noise_norm=1, constellation=1, guard=guard)


def sys_of(p, precision=0):
    return W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift, bits=p.bits,
                  S=p.S, noise_norm=p.noise_norm, constellation=p.constellation, precision=precision, guard=p.guard)


def masked_tx_stream(p, v_tx, sym_idx, roll_off=10):
    """The Tx half of the oracle's frame_chain_masked: sym_idx (N, S) -> the serialised stream of tail_tx + S stride
    samples (gen_tx_ofdm, dft_rc_filt and tx2rx, main_channel_mask.m:384-431), built from the oracle's own pieces.
    roll_off=None: the same symbols without the mask (the unmasked guard-band stream)."""
    X = np.where(p.active[:, None], O.qam_points(p.bits, p.constellation)[sym_idx], 0.0)
    x = np.fft.ifft(X, axis=0)
    t = v_tx[:, None] * x[(np.arange(p.n_tx) - p.cp) % p.N, :]                # (n_tx, S)
    if roll_off is not None:
        t = O.mask_symbols(t, roll_off)
    u = np.zeros(p.tail_tx + p.S * p.stride, dtype=np.complex128)
    for s in range(p.S):
        u[s * p.stride: s * p.stride + p.n_tx] += t[:, s]
    return u


def psd_estimate_hann(x, fft_len):
    """Estimator 1 of wofdm_psd_masked: slices of fft_len samples at a hop of fft_len / 2 (no remainder slice), taper
    w[n] = sin^2(pi n / fft_len), |fftshift(fft)|^2 averaged over the slices and scaled by fft_len / sum(w^2) = 8/3, so a
    white stream reads the level of the oracle's psd_estimate.  Needs len(x) >= fft_len."""
    hop = fft_len // 2
    n = (len(x) - fft_len) // hop + 1
    w = np.sin(np.pi * np.arange(fft_len) / fft_len) ** 2
    acc = np.zeros(fft_len)
    for k in range(n):
        acc += np.abs(np.fft.fftshift(np.fft.fft(w * x[k * hop: k * hop + fft_len]))) ** 2
    return acc * (fft_len / np.sum(w ** 2)) / n


def oracle_psd(p, vt, sym, roll_off, estimator):
    """mean over frames sym (F, S, N) of the estimator's PSD of the masked and the unmasked stream"""
    est = O.psd_estimate if estimator == "reference" else psd_estimate_hann
    P = 8 * p.N
    m = np.mean([est(masked_tx_stream(p, vt, s.T, roll_off), P) for s in sym], axis=0)
    u = np.mean([est(masked_tx_stream(p, vt, s.T, None), P) for s in sym], axis=0)
    return m, u


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_parseval_of_both_estimators():
    rng = np.random.default_rng(3)
    P = 1024
    for n in (P, 3 * P, 3 * P + 517):
        x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
        ref = O.psd_estimate(x, P)                     # floor(n / P) + 1 slices that partition x (last zero padded)
        assert abs(ref.sum() * (n // P + 1) / (P * np.vdot(x, x).real) - 1) < 1e-12
        hop = P // 2
        ns = (n - P) // hop + 1
        w = np.sin(np.pi * np.arange(P) / P) ** 2
        energy = sum(np.sum(np.abs(w * x[k * hop: k * hop + P]) ** 2) for k in range(ns))
        assert abs(psd_estimate_hann(x, P).sum() * ns / (8 / 3) / (P * energy) - 1) < 1e-12
    # a white stream reads the same level under both
    x = rng.standard_normal(200 * P) + 1j * rng.standard_normal(200 * P)
    assert abs(psd_estimate_hann(x, P).mean() / O.psd_estimate(x, P).mean() - 1) < 0.02


@pytest.mark.parametrize("name,N,cp,ttx,trx,guard,S,roll_off", [
    ("wtx", 256, 16, 8, 0, 64, 5, 10), ("CPW", 128, 8, 4, 4, 20, 4, 30), ("WOLA", 512, 32, 16, 16, 128, 3, 10)])
def test_masked_tx_stream(name, N, cp, ttx, trx, guard, S, roll_off):
    """masked_tx_stream is the oracle's frame_chain_masked Tx stream and the serialisation of the product form's symbols; with
    roll_off=None it is the unmasked guard-band stream built from qam_points and an IDFT."""
    p = chain_params(name, N, cp, ttx, trx, guard, S)
    rng = np.random.default_rng(7)
    vt = O.perturbed_windows(p, seed=2)[0]
    sym = rng.integers(0, 16, size=(N, S))
    u = masked_tx_stream(p, vt, sym, roll_off)
    nz = rng.standard_normal(O.noise_len(p, 3)) + 0j
    r = O.frame_chain_masked(p, vt, O.rc_window_rx(p), np.array([1.0, 0.2, 0.1]), 30.0, sym, nz, roll_off=roll_off)
    assert np.array_equal(u, r.tx_stream)

    def serialise(t):
        out = np.zeros(p.tail_tx + S * p.stride, dtype=complex)
        for s in range(S):
            out[s * p.stride: s * p.stride + p.n_tx] += t[:, s]
        return out
    X = np.where(p.active[:, None], O.qam_points(p.bits, p.constellation)[sym], 0.0)
    a = X[(np.arange(p.N - 2 * guard) + guard + N // 2) % N]                          # active bins in centred order
    f = O.mask_symbols_product(p, vt, a, roll_off)
    assert np.max(np.abs(u - serialise(f))) < 1e-12 * np.max(np.abs(u))
    x = np.fft.ifft(X, axis=0)
    t = vt[:, None] * x[(np.arange(p.n_tx) - cp) % N]
    assert np.array_equal(masked_tx_stream(p, vt, sym, None), serialise(t))


def test_obr_split_of_the_mirror():
    x = np.arange(2048, dtype=float)
    obr, mf = U.obr_split(x, 64)
    gb = 512
    assert obr == pytest.approx(np.mean(np.r_[x[:gb], x[-gb:]]))
    assert np.array_equal(mf, x[gb:2048 - gb])
    with pytest.raises(ValueError):
        U.obr_split(x, 0)


def test_handle_checks_the_window_before_the_call():
    h = W.Handle.__new__(W.Handle)          # (no device needed: the check runs before the library is called)
    h._h = None
    s = W.SysT(N=256, cp=16, cs=8, tail_tx=8, bits=4, S=16, constellation=1, guard=64)
    with pytest.raises(W.WofdmError) as e:
        h.psd_masked(s, np.ones(279))
    assert e.value.code == capi.EINVAL
    with pytest.raises(W.WofdmError) as e:
        h.psd_masked(s, np.ones(280), estimator="welch")
    assert e.value.code == capi.EINVAL


# ---- GPU ---------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def handle():
    h = W.Handle([0])
    yield h
    h.close()


# (name, N, cp, tail_tx, tail_rx, guard, S, roll_off, f0, frames)
REPLAY = [
    ("wtx", 128, 8, 4, 0, 32, 16, 10, 0, 6),
    ("wtx", 256, 16, 8, 0, 64, 16, 10, 5, 6),          # bench.py's mask_chain shape
    ("wtx", 256, 16, 8, 0, 64, 256, 30, 0, 2),
    ("CPW", 256, 16, 8, 8, 64, 16, 30, 100, 4),
    ("WOLA", 512, 32, 16, 16, 128, 64, 10, 7, 3),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,cp,ttx,trx,guard,S,roll_off,f0,F", REPLAY)
def test_replay_against_the_oracle(handle, name, N, cp, ttx, trx, guard, S, roll_off, f0, F):
    """Production frames exported with wofdm_ber_draws (same sys and seed), both oracle streams, both estimators, bin by
    bin.  Tolerance from the product's known error (Tx streams within 2e-6 of their peak, fp16 hi + lo operands, fp32
    accumulation): a bin's amplitude error is then about 1e-5 of the in-band level, so |X|^2 is good to ~2e-5 relative in
    band and ~2e-3 relative 40 dB below it; bins further down are held to that absolute floor."""
    p = chain_params(name, N, cp, ttx, trx, guard, S)
    s = sys_of(p)
    vt = O.perturbed_windows(p, seed=5)[0]
    seed = 11
    sym, _ = handle.ber_draws(s, 1, seed, 0, np.arange(f0, f0 + F))
    for estimator in ("reference", "hann"):
        dm, du = handle.psd_masked(s, vt, roll_off=roll_off, frames=F, f0=f0, seed=seed, estimator=estimator)
        om, ou = oracle_psd(p, vt, sym, roll_off, estimator)
        for got, ref, what in ((dm, om, "masked"), (du, ou, "unmasked")):
            inband = ref[8 * guard: 8 * (N - guard)].mean()
            dev = np.abs(got - ref) / (ref + 1e-4 * inband)
            print(f"{name} N={N} S={S} roll-off {roll_off} {estimator} {what}: worst deviation {dev.max():.2e} "
                  f"(relative to the bin + 1e-4 x in-band)")
            assert dev.max() < 4e-3, (what, estimator, int(np.argmax(dev)), dev.max())


@pytest.mark.gpu
def test_ranges_add_up_and_do_not_depend_on_the_batch(handle):
    """More frames than one product batch (S = 256: 512 frames per batch): [0, a) and [a, b) weighted by their frame
    counts give [0, b); the masked half does not depend on whether the unmasked one is asked for; same seed, same result;
    another seed, another result."""
    p = chain_params(S=256)
    s = sys_of(p)
    vt = O.rc_window_tx(p)
    a, b = 500, 1200
    for est in ("reference", "hann"):
        fm, fu = handle.psd_masked(s, vt, frames=b, seed=4, estimator=est)
        am, au = handle.psd_masked(s, vt, frames=a, seed=4, estimator=est)
        bm, bu = handle.psd_masked(s, vt, frames=b - a, f0=a, seed=4, estimator=est)
        np.testing.assert_allclose((a * am + (b - a) * bm) / b, fm, rtol=1e-12, atol=0)
        np.testing.assert_allclose((a * au + (b - a) * bu) / b, fu, rtol=1e-12, atol=0)
        only_m, none_u = handle.psd_masked(s, vt, frames=b, seed=4, estimator=est, unmasked=False)
        none_m, only_u = handle.psd_masked(s, vt, frames=b, seed=4, estimator=est, masked=False)
        assert none_u is None and none_m is None
        np.testing.assert_allclose(only_m, fm, rtol=1e-12, atol=0)
        np.testing.assert_allclose(only_u, fu, rtol=1e-12, atol=0)
        again_m, again_u = handle.psd_masked(s, vt, frames=b, seed=4, estimator=est)
        np.testing.assert_allclose(again_m, fm, rtol=1e-12, atol=0)
        np.testing.assert_allclose(again_u, fu, rtol=1e-12, atol=0)
        other_m, _ = handle.psd_masked(s, vt, frames=b, seed=5, estimator=est)
        assert not np.allclose(other_m, fm, rtol=1e-6, atol=0)


@pytest.mark.gpu
def test_ensemble_levels_agree_with_the_oracle(handle):
    """What the call exists for: Hann estimator, many frames at the mask_chain shape; the device's OBR, deep out-of-band
    (more than 32 sub-carriers from the band edge) and in-band levels of both streams against the oracle's average over
    numpy draws, within the Monte-Carlo error."""
    p = chain_params(S=256)
    s = sys_of(p)
    vt = O.rc_window_tx(p)
    dm, du = handle.psd_masked(s, vt, roll_off=10, frames=400, seed=9, estimator="hann")
    rng = np.random.default_rng(0)
    sym = rng.integers(0, 16, size=(16, p.S, p.N))
    om, ou = oracle_psd(p, vt, sym, 10, "hann")
    gb, P = 8 * p.guard, 8 * p.N
    band = slice(gb + 16, P - gb - 16)
    deep = np.r_[0:gb - 256, P - gb + 256:P]
    for got, ref, what in ((dm, om, "masked"), (du, ou, "unmasked")):
        inb_d, inb_o = got[band].mean(), ref[band].mean()
        obr_d, obr_o = U.obr_split(got, p.guard)[0], U.obr_split(ref, p.guard)[0]
        deep_d, deep_o = got[deep].mean(), ref[deep].mean()
        print(f"{what}: OBR {10 * np.log10(obr_d / inb_d):.1f} dB (oracle {10 * np.log10(obr_o / inb_o):.1f}), deep "
              f"out-of-band {10 * np.log10(deep_d / inb_d):.1f} dB (oracle {10 * np.log10(deep_o / inb_o):.1f})")
        assert abs(inb_d / inb_o - 1) < 0.02, what
        assert abs(obr_d / obr_o - 1) < 0.10, what
        assert abs(deep_d / deep_o - 1) < 0.10, what


def _raw(handle, s, vt, roll_off=10, seed=0, f0=0, n=2, est=0, m=True, u=True):
    P = 8 * s.N
    om = np.empty(P) if m else None
    ou = np.empty(P) if u else None
    return capi.load().wofdm_psd_masked(handle._h, C.byref(s), vt.ctypes.data_as(capi._dp) if vt is not None else None,
                                        roll_off, seed, f0, n, est, om.ctypes.data_as(capi._dp) if m else None,
                                        ou.ctypes.data_as(capi._dp) if u else None)


@pytest.mark.gpu
def test_rejections_leave_the_handle_usable(handle):
    p = chain_params()
    s = sys_of(p)
    vt = O.rc_window_tx(p)
    E, U_ = capi.EINVAL, capi.EUNSUPPORTED
    big = chain_params(guard=0, S=1024)
    p1024 = chain_params(N=1024, guard=256)
    cases = [
        (E, dict(vt=None)),
        (E, dict(m=False, u=False)),
        (E, dict(f0=-1)),
        (E, dict(n=0)),
        (E, dict(f0=2 ** 63 - 2, n=5)),
        (E, dict(est=2)),
        (E, dict(roll_off=0)),
        (E, dict(roll_off=1000)),
        (E, dict(s=sys_of(chain_params(S=2)))),                    # 8 + 2 * 272 < 2048 samples
        (U_, dict(s=sys_of(p, precision=1))),
        (U_, dict(s=sys_of(p1024), vt=O.rc_window_tx(p1024))),
        (U_, dict(s=sys_of(chain_params(bits=8)))),                # a guard band needs bits < 8
        (U_, dict(s=sys_of(big), vt=O.rc_window_tx(big))),         # the symbol kernel cannot hold 1024 symbols of 256 bins
    ]
    for code, kw in cases:
        kw.setdefault("s", s)
        kw.setdefault("vt", vt)
        assert _raw(handle, **kw) == code, kw
        assert _raw(handle, s, vt) == 0, kw
    dm, du = handle.psd_masked(s, vt, frames=2)
    assert np.all(np.isfinite(dm)) and np.all(du > 0)


@pytest.mark.gpu
def test_psd_sim_mc_mirror(handle):
    p = chain_params()
    vt = O.rc_window_tx(p)
    r = U.psd_sim_mc(8, p.cp, p.cs, p.tail_tx, np.diag(vt), p.guard, p.N, p.bits, p.S, 10, seed=3, handle=handle)
    assert set(r) == {"X_est_masked", "X_est", "obr_masked", "obr", "mf_band_masked", "mf_band", "f_axis"}
    for k in ("X_est_masked", "X_est", "f_axis"):
        assert r[k].shape == (2048,)
    assert r["mf_band"].shape == r["mf_band_masked"].shape == (2048 - 2 * 512,)
    assert r["f_axis"][0] == -0.5 and r["f_axis"][1024] == 0.0
    s = sys_of(p)
    xm, xu = handle.psd_masked(s, vt, roll_off=10, frames=8, seed=3)
    np.testing.assert_allclose(r["X_est_masked"], xm, rtol=1e-12)
    np.testing.assert_allclose(r["X_est"], xu, rtol=1e-12)
    assert r["obr"] == pytest.approx(U.obr_split(xu, p.guard)[0])
    with pytest.raises(ValueError):
        U.psd_sim_mc(8, p.cp, p.cs, p.tail_tx, vt, 0, p.N, p.bits, p.S, 10, handle=handle)
