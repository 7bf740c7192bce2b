"""The channel-mask chain's counters resolved by sub-carrier and by channel, and its shards (wofdm_ber_run_masked_resolved,
wofdm_ber_run_masked_shard).

GPU: summed over the cells, the resolved counters are wofdm_ber_run_masked's, bit for bit, on every kernel the masked chain
runs (the resolved call runs that kernel's twin; each row checks both names); every (SNR, channel, bin) cell against the
oracle's masked chain on replayed draws; guard bins and totals; shards and batches that do not move a counter; errors; the
run_sim_mc mirror.
"""
import ctypes as C
import re

import numpy as np
import pytest

import wofdm_b200 as W
from oracle import ber_resolved as R
from oracle import wofdm_oracle as O

RESOLVE = [(True, False), (False, True), (True, True)]     # (by_subcarrier, by_channel)
ENV = ("WOFDM_DEBUG", "WOFDM_MASK_FFT", "WOFDM_MASK_DUMP", "WOFDM_RESOLVED_STAGED", "WOFDM_NO_TCONV", "WOFDM_VARIANT")


@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


@pytest.fixture
def clean_env(monkeypatch):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def to_sys(p):
    return W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift, bits=p.bits,
                  S=p.S, noise_norm=p.noise_norm, constellation=p.constellation, precision=0, guard=p.guard)


def kernels_of(fn, monkeypatch, capfd):
    """(fn(), names of the K1 kernels it prepared) -- the WOFDM_DEBUG residency report of prepare_kernel."""
    monkeypatch.setenv("WOFDM_DEBUG", "1")
    capfd.readouterr()
    try:
        out = fn()
    finally:
        monkeypatch.delenv("WOFDM_DEBUG")
    names = set(re.findall(r"\[wofdm\] (\S+): smem \d+ B, \d+ CTAs/SM", capfd.readouterr().err))
    return out, names


def one(names):
    assert len(names) == 1, names
    return next(iter(names))


# (system, N, cp, tail_tx, tail_rx, bits, S, L, guard, WOFDM_MASK_FFT, production kernel, twin)  -- full-name patterns
CASES = {
    "gather_n256": ("wtx", 256, 16, 8, 0, 4, 16, 21, 64, False, r"ber_f32t2_n256_t256_tiles\d+_b2_txy", r"ber_f32t2_n256_t256_tiles\d+_b2_txy_res"),
    "gather_n512": ("CPW", 512, 32, 16, 20, 4, 16, 21, 128, False, r"ber_f32t2_n512_t512_tiles\d+_b1_txy", r"ber_f32t2_n512_t512_tiles\d+_b1_txy_res"),
    # S < 8: too few samples for the tensor-core kernel's tiles -> the register kernel on the assembled stream
    "regs_txs_wola_s7": ("WOLA", 256, 30, 8, 10, 4, 7, 21, 64, False, r"ber_f32r_n256_t256_c\d+_l21_b2_f(true|false)_txs", r"ber_f32r_n256_t256_c\d+_l21_b2_f(true|false)_txs_res"),
    "staged_cp_n128": ("CP", 128, 8, 0, 0, 2, 16, 21, 0, False, r"ber_f32_n128_t128_c0_l0_b1_ffalse", r"ber_f32_n128_t128_c0_l0_b1_f0_res"),
    # 48 symbols: more than one Tx pass of the tuned kernels -> staged
    "staged_wtx_s48": ("wtx", 256, 16, 8, 0, 4, 48, 21, 0, False, r"ber_f32_n256_t256_c0_l0_b1_ffalse", r"ber_f32_n256_t256_c0_l0_b1_f0_res"),
    # 30 taps: the gather kernels hold 21; the tensor-core kernel of 84 taps on the assembled stream
    "tconv2_l84_wtx_l30": ("wtx", 256, 16, 8, 0, 4, 16, 30, 64, False, r"ber_f32t2_n256_t256_tiles\d+_b2_cl1_l84", r"ber_f32t2_n256_t256_tiles\d+_b2_cl1_l84_res"),
    # WOFDM_MASK_FFT=1: the per-symbol FFT kernel writes the assembled stream, the tensor-core kernel reads it
    "mask_fft_n256": ("wtx", 256, 16, 8, 0, 4, 16, 21, 64, True, r"ber_f32t2_n256_t256_tiles\d+_b2", r"ber_f32t2_n256_t256_tiles\d+_b2_cl1_lTCV_LB_res"),
}


def case_setup(case):
    name, N, cp, ttx, trx, bits, S, L, guard, fft, kp, kt = CASES[case]
    p = O.system_params(name, N, cp, ttx, trx, S=S, bits=bits, noise_norm=1, constellation=1, guard=guard)
    vt, vr, _, _ = O.perturbed_windows(p, seed=N + cp)
    return p, to_sys(p), vt, vr, L, fft, kp, kt


def frames_per_cell(n_snr, C_, ens, shard=(0, 1)):
    total = n_snr * C_ * ens
    lo, hi = total * shard[0] // shard[1], total * (shard[0] + 1) // shard[1]
    f = np.arange(lo, hi)
    return np.bincount(f // ens, minlength=n_snr * C_).reshape(n_snr, C_)


def check_cells_and_totals(p, r, fpc, chan):
    """Guard bins are zero in every array; sym_tot = frames of the cell x (S - 1) on active bins; bit_tot = sym_tot x bits."""
    cells = fpc if chan else fpc.sum(axis=1, keepdims=True)
    if r["sym_tot"].shape[2] > 1:
        act = p.active
        assert np.array_equal(r["sym_tot"][:, :, act], np.broadcast_to(cells[:, :, None] * (p.S - 1), r["sym_tot"][:, :, act].shape))
        for key in ("sym_tot", "bit_tot", "sym_err", "bit_err"):
            assert not r[key][:, :, ~act].any(), key
    else:
        assert np.array_equal(r["sym_tot"][:, :, 0], cells * int(np.count_nonzero(p.active)) * (p.S - 1))
    assert np.array_equal(r["bit_tot"], r["sym_tot"] * p.bits)
    assert np.all(r["sym_err"] <= r["bit_err"]) and np.all(r["sym_err"] <= r["sym_tot"])


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_sum_identity(handle, case, clean_env, capfd):
    """For every resolve value, the resolved counters summed over the cells equal ber_run_masked's bit for bit, and the
    call ran the twin of the kernel the unresolved call ran."""
    p, s, vt, vr, L, fft, kp, kt = case_setup(case)
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    chans = O.synth_channels(3, L, seed=p.N + L)
    snr = np.array([6.0, 12.0, 18.0]) + (0.0 if p.bits > 2 else -6.0)
    ens = 5
    kw = dict(seed=p.N + p.cp, variant=1, roll_off=10)
    ref, kref = kernels_of(lambda: handle.ber_run_masked(s, vt, vr, chans, snr, ens, **kw), clean_env, capfd)
    assert re.fullmatch(kp, one(kref)), (case, kref)
    assert ref["sym_err"].sum() > 0, "a sum identity over zero errors proves nothing"
    fpc = frames_per_cell(len(snr), 3, ens)
    out = {}
    for bins, chan in RESOLVE:
        r, kres = kernels_of(lambda: handle.ber_run_masked_resolved(s, vt, vr, chans, snr, ens, by_subcarrier=bins,
                                                                    by_channel=chan, **kw), clean_env, capfd)
        assert re.fullmatch(kt, one(kres)), (case, kres)
        cr, nr = (3 if chan else 1), (p.N if bins else 1)
        for key in ("bit_err", "sym_err", "sym_tot", "bit_tot"):
            assert r[key].shape == (len(snr), cr, nr), key
        for key in ("bit_err", "sym_err", "sym_tot", "bit_tot"):
            assert np.array_equal(r[key].sum(axis=(1, 2)), ref[key]), (case, bins, chan, key, r[key].sum(axis=(1, 2)), ref[key])
        check_cells_and_totals(p, r, fpc, chan)
        out[(bins, chan)] = r
    both = out[(True, True)]
    assert np.array_equal(both["sym_err"].sum(axis=2), out[(False, True)]["sym_err"][..., 0])
    assert np.array_equal(both["bit_err"].sum(axis=1), out[(True, False)]["bit_err"][:, 0, :])


def dist(v, m):
    b = np.arange(-(m - 2), m - 1, 2.0)
    return np.min(np.abs(v[..., None] - b), axis=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("fft", [False, True])
def test_cells_match_oracle(handle, fft, clean_env):
    """2 SNR points x 3 channels x ensemble 2: every frame replayed from its exported draws through the oracle's masked
    chain (frame_chain_masked, fp64), every (SNR, channel, bin) cell within its boundary-flip slack.  A decision counts as
    near a boundary when the oracle's equalised value lies within 1e-3 x max(1, |x|) lattice units of one -- ten times the
    band of the unmasked fp32 chain (test_ber_resolved.cells_vs_oracle), because the masked Tx stream of the device is only
    within 8e-6 of its peak of the FFT kernel's (test_drivers_gpu), several times the fp32 rounding of the plain chain."""
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    L = 21
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    vt, vr, _, _ = O.perturbed_windows(p, seed=5)
    chans = O.synth_channels(3, L, seed=9)
    snr = np.array([8.0, 16.0])
    ens = 2
    r = handle.ber_run_masked_resolved(s, vt, vr, chans, snr, ens, seed=21, variant=1, roll_off=10, by_subcarrier=True,
                                       by_channel=True)
    F = len(snr) * 3 * ens
    sym, nz = handle.ber_draws(s, L, 21, 1, np.arange(F))
    want_s = np.zeros((2, 3, p.N), dtype=np.int64)
    want_b = np.zeros((2, 3, p.N), dtype=np.int64)
    slack = np.zeros((2, 3, p.N), dtype=np.int64)
    m, sc = O.qam_levels(p.bits), O.qam_scale(p.bits, p.constellation)
    for f in range(F):
        si, c = f // (3 * ens), (f // ens) % 3
        res = O.frame_chain_masked(p, vt, vr, chans[:, c], snr[si], sym[f].T, nz[f], roll_off=10)
        a, b = R.per_bin_errors(p, res, sym[f].T)
        want_s[si, c] += a
        want_b[si, c] += b
        x = res.eq / sc
        near = np.minimum(dist(x.real, m), dist(x.imag, m)) <= 1e-3 * np.maximum(1.0, np.abs(x))
        slack[si, c] += near.sum(axis=1)
    got_s, got_b = r["sym_err"], r["bit_err"]
    assert want_s.sum() > 0
    assert np.all(np.abs(got_s - want_s) <= slack), (np.abs(got_s - want_s).max(), slack.max())
    assert np.all(np.abs(got_b - want_b) <= 2 * slack), (np.abs(got_b - want_b).max(), slack.max())
    assert not r["sym_err"][..., ~p.active].any()


@pytest.mark.gpu
@pytest.mark.parametrize("fft", [False, True])
def test_shards_and_batches_do_not_move_a_counter(handle, fft, clean_env):
    """17 000 frames: more than one batch of the mask product (16 384; 8 192 for the FFT kernel), and with ensemble 1 700
    every CTA of the ~300 in flight crosses cells within a launch.  1, 2, 3 and 47 shards -- every one its own batches,
    launches and flushes -- add up with no tolerance: for ber_run_masked and, cell by cell, for the resolved counters."""
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    vt, vr, _, _ = O.perturbed_windows(p, seed=3)
    chans = O.synth_channels(5, 21, seed=6)
    snr = np.array([4.0, 10.0])
    ens = 1700
    kw = dict(seed=17, variant=1, roll_off=10)
    full = handle.ber_run_masked(s, vt, vr, chans, snr, ens, **kw)
    fres = handle.ber_run_masked_resolved(s, vt, vr, chans, snr, ens, by_subcarrier=True, by_channel=True, **kw)
    assert full["sym_err"].sum() > 10 ** 5
    for key in ("bit_err", "sym_err", "bit_tot", "sym_tot"):
        assert np.array_equal(fres[key].sum(axis=(1, 2)), full[key]), key
    for W_ in (2, 3, 47):
        acc = {key: np.zeros_like(full[key]) for key in full}
        racc = {key: np.zeros_like(fres[key]) for key in fres}
        for k in range(W_):
            part = handle.ber_run_masked(s, vt, vr, chans, snr, ens, shard=(k, W_), **kw)
            rpart = handle.ber_run_masked_resolved(s, vt, vr, chans, snr, ens, shard=(k, W_), by_subcarrier=True,
                                                   by_channel=True, **kw)
            check_cells_and_totals(p, rpart, frames_per_cell(2, 5, ens, (k, W_)), True)
            for key in acc:
                acc[key] += part[key]
            for key in racc:
                racc[key] += rpart[key]
        for key in acc:
            assert np.array_equal(acc[key], full[key]), (W_, key, acc[key], full[key])
        for key in racc:
            assert np.array_equal(racc[key], fres[key]), (W_, key, np.argwhere(racc[key] != fres[key])[:5])


@pytest.mark.gpu
def test_two_device_handle_matches_one_device(handle, clean_env):
    n = C.c_int(0)
    assert W.capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("one visible device")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    vt, vr, _, _ = O.perturbed_windows(p, seed=1)
    chans = O.synth_channels(3, 21, seed=2)
    kw = dict(seed=3, variant=1, roll_off=10)
    one_ = handle.ber_run_masked_resolved(s, vt, vr, chans, [4.0, 8.0], 300, by_channel=True, **kw)
    sh = handle.ber_run_masked(s, vt, vr, chans, [4.0, 8.0], 300, shard=(1, 3), **kw)
    with W.Handle([0, 1]) as h2:
        two = h2.ber_run_masked_resolved(s, vt, vr, chans, [4.0, 8.0], 300, by_channel=True, **kw)
        sh2 = h2.ber_run_masked(s, vt, vr, chans, [4.0, 8.0], 300, shard=(1, 3), **kw)
    for key in one_:
        assert np.array_equal(one_[key], two[key]), key
    for key in sh:
        assert np.array_equal(sh[key], sh2[key]), key


@pytest.mark.gpu
def test_errors_and_handle_survives(handle, clean_env):
    s = W.params_from_name("CP", 128, 8, 0, 0, bits=4, S=4, noise_norm=1, constellation=1)
    vt, vr = np.ones(s.n_tx), np.ones(s.N)
    chans = O.synth_channels(2, 5, seed=2)
    lib = W.capi.load()
    ch = np.ascontiguousarray(np.stack([chans.real.T, chans.imag.T], axis=-1), dtype=np.float64)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    snr = np.array([5.0])
    out = [np.zeros(2 * 128, dtype=np.int64) for _ in range(4)]

    def resolved(resolve, ptrs, sys=s, n_snr=1, snr_arr=snr, shard=(0, 1), roll_off=10, wt=vt, wr=vr, n_chan=2):
        return lib.wofdm_ber_run_masked_resolved(handle._h, C.byref(sys), dp(wt), dp(wr), dp(ch), 5, n_chan, dp(snr_arr), n_snr, 2,
                                                 0, 1, roll_off, shard[0], shard[1], resolve, *ptrs)

    def sharded(ptrs, shard=(0, 1), sys=s, roll_off=10):
        return lib.wofdm_ber_run_masked_shard(handle._h, C.byref(sys), dp(vt), dp(vr), dp(ch), 5, 2, dp(snr), 1, 2, 0, 1,
                                              roll_off, shard[0], shard[1], *ptrs)

    ref = handle.ber_run_masked(s, vt, vr, chans, snr, 2, seed=0, variant=1)

    def still_works():
        r = handle.ber_run_masked_resolved(s, vt, vr, chans, snr, 2, seed=0, variant=1, by_channel=True)
        for key in ref:
            assert np.array_equal(r[key].sum(axis=(1, 2)), ref[key]), key

    ok3 = [ip(o) for o in out[:3]]
    for resolve in (0, 4, 5, -1):
        assert resolved(resolve, ok3) == W.capi.EINVAL
    for k in range(3):
        ptrs = list(ok3)
        ptrs[k] = None
        assert resolved(1, ptrs) == W.capi.EINVAL
    for k in range(4):
        ptrs = [ip(o) for o in out]
        ptrs[k] = None
        assert sharded(ptrs) == W.capi.EINVAL
    for bad in ((-1, 2), (2, 2), (0, 0), (3, 1)):
        assert resolved(1, ok3, shard=bad) == W.capi.EINVAL
        assert sharded([ip(o) for o in out], shard=bad) == W.capi.EINVAL
    still_works()
    # 2^30 points x 2^30 channels x 128 bins x 16 bytes of counters overflow size_t (the check reads no input array)
    assert resolved(3, ok3, n_snr=1 << 30, snr_arr=np.zeros(1), n_chan=1 << 30) == W.capi.EINVAL
    # 2^26 points x 2 channels x 128 bins x 16 bytes = 256 GiB of device counters, more than the card holds: the device
    # buffer fails before any host counter array is allocated
    big = np.full(1 << 26, 5.0)
    assert resolved(3, ok3, n_snr=1 << 26, snr_arr=big) == W.capi.ENOMEM
    still_works()
    # what wofdm_ber_run_masked rejects: fp64, N outside {128, 256, 512}, roll_off, n_tx > 1.5 N
    assert resolved(1, ok3, sys=s.copy(precision=1)) == W.capi.EUNSUPPORTED
    assert sharded([ip(o) for o in out], sys=s.copy(precision=1)) == W.capi.EUNSUPPORTED
    s64 = W.params_from_name("CP", 64, 8, 0, 0, bits=4, S=4, noise_norm=1, constellation=1)
    assert resolved(1, ok3, sys=s64, wt=np.ones(s64.n_tx), wr=np.ones(64)) == W.capi.EUNSUPPORTED
    assert resolved(1, ok3, roll_off=0) == W.capi.EINVAL
    assert sharded([ip(o) for o in out], roll_off=0) == W.capi.EINVAL
    slong = W.params_from_name("CP", 128, 80, 0, 0, bits=4, S=4, noise_norm=1, constellation=1)
    assert resolved(1, ok3, sys=slong, wt=np.ones(slong.n_tx)) == W.capi.EUNSUPPORTED
    still_works()
    # more shards than frames: empty shards count nothing, the others add up
    parts = [handle.ber_run_masked(s, vt, vr, chans, snr, 2, seed=0, variant=1, shard=(k, 7)) for k in range(7)]
    for key in ref:
        assert np.array_equal(sum(q[key] for q in parts), ref[key]), key


@pytest.mark.gpu
def test_run_sim_mc_per_subcarrier_mirror(handle, clean_env):
    """The mean of run_sim_mc_per_subcarrier over the active bins is run_sim_mc's [berMasked, ber], for the same seed."""
    from wofdm_b200 import ofdm_utils as U
    for name, cp, ttx, trx in (("wtx", 16, 8, 0), ("WOLA", 22, 8, 10)):
        p = O.system_params(name, 256, cp, ttx, trx, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
        vt, vr, _, _ = O.perturbed_windows(p, seed=cp)
        ch = O.synth_channels(1, 21, seed=cp)[:, 0]
        args = (7, p.cp, p.cs, ttx, trx, np.diag(vt), np.diag(vr), ch, 12.0, 64, p.rm, p.shift, 256, 4, 16, 10)
        bm, b0 = U.run_sim_mc(*args, seed=3, handle=handle)
        pm, p0 = U.run_sim_mc_per_subcarrier(*args, seed=3, handle=handle)
        assert pm.shape == p0.shape == (256,)
        assert not pm[~p.active].any() and not p0[~p.active].any()
        assert pm[p.active].mean() == pytest.approx(bm, rel=1e-12, abs=0)
        assert p0[p.active].mean() == pytest.approx(b0, rel=1e-12, abs=0)
        assert bm > 0 and b0 > 0
