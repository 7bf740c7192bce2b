"""Error counters resolved by sub-carrier and by channel realisation (wofdm_ber_run_resolved).

CPU: the oracle's per-bin counts (oracle/ber_resolved.py) add up to the golden frames' pinned counts.
GPU: summed over the channel and bin axes the resolved counters are wofdm_ber_run_multi's, bit for bit, on every policy
production picks (the resolved call runs that kernel's twin); every (SNR, channel, bin) cell against the oracle on replayed
draws, also for the staged fallback with production's noise numbering; totals, guard bins, sharding, errors, and the
wOFDMSystem mirror.
"""
import ctypes as C

import numpy as np
import pytest

import wofdm_b200 as W
from oracle import ber_resolved as R
from oracle import wofdm_oracle as O
from helpers import golden_params, golden_windows, load_ser_golden, replay_frames

RESOLVE = [(True, False), (False, True), (True, True)]     # (by_subcarrier, by_channel)


# ---------------------------------------------------------------- CPU

@pytest.mark.parametrize("name", O.SYSTEMS)
def test_oracle_per_bin_counts_sum_to_golden_frames(name):
    """Case B of the golden vectors (one frame per SNR value, counts pinned by the reference): the per-bin counts of the
    python convention sum to the pinned symbol errors and to the frame's bit errors; the same frames in the MATLAB Gray
    convention (indices converted, same lattice points) sum to that frame's own counts."""
    g = load_ser_golden(name)
    p = golden_params(g, g["B_S"])
    wins = golden_windows(g, p)
    for i, snr in enumerate(g["B_snr"]):
        fr = replay_frames(p, wins, g["B_channels"], 1, [snr], int(g["B_seed"][i]))[0]
        for w, (vt, vr) in enumerate(wins):
            res = O.frame_chain_structured(p, vt, vr, fr["chan"], fr["snr"], fr["sym_idx"], fr["noise"][w])
            sym, bit = R.per_bin_errors(p, res, fr["sym_idx"])
            assert sym.shape == (p.N,) and bit.shape == (p.N,)
            assert int(sym.sum()) == int(round(g["B_ser"][i][w] * p.N * (p.S - 1))) == res.sym_err
            assert int(bit.sum()) == res.bit_err and np.all(bit >= sym)
            # MATLAB Gray: the same lattice points, indexed and bit-mapped the MATLAB way
            pg = golden_params(g, g["B_S"], constellation=1)
            idx_g = R.convert_indices(fr["sym_idx"], p.bits, 0, 1)
            scale = O.qam_scale(p.bits, 1)
            rg = O.frame_chain_structured(pg, vt, vr, fr["chan"], fr["snr"], idx_g, fr["noise"][w] * scale)
            sg, bg = R.per_bin_errors(pg, rg, idx_g)
            assert int(sg.sum()) == rg.sym_err and int(bg.sum()) == rg.bit_err


def test_oracle_per_bin_counts_guard_band():
    """Null bins of a guard band count nothing."""
    p = O.system_params("WOLA", 64, 8, 4, 4, S=4, bits=4, guard=16)
    vt, vr, _, _ = O.perturbed_windows(p, seed=3)
    rng = np.random.default_rng(0)
    h = O.synth_channels(1, 5, seed=1)[:, 0]
    n = O.noise_len(p, 5)
    sym_idx = rng.integers(0, 16, size=(64, 4))
    res = O.frame_chain_structured(p, vt, vr, h, -5.0, sym_idx, rng.standard_normal(n) + 1j * rng.standard_normal(n))
    s, b = R.per_bin_errors(p, res, sym_idx)
    assert np.all(s[~p.active] == 0) and np.all(b[~p.active] == 0)
    assert int(s.sum()) == res.sym_err > 0 and int(b.sum()) == res.bit_err


# ---------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def to_sys(p, precision):
    return W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift,
                  bits=p.bits, S=p.S, noise_norm=p.noise_norm, constellation=p.constellation, precision=precision,
                  guard=p.guard)


def frames_per_cell(n_snr, C, ens, shard=(0, 1)):
    f = np.arange(n_snr * C * ens)
    f = f[f % shard[1] == shard[0]]
    return np.bincount(f // ens, minlength=n_snr * C).reshape(n_snr, C)


def check_sum_identity(handle, p, s, wins, chans, snr, ens, seed=7, variant=0):
    """Every resolution against wofdm_ber_run_multi, bit for bit, plus the totals; returns the (bins x channels) result."""
    wt, wr = [w[0] for w in wins], [w[1] for w in wins]
    ref = handle.ber_run_multi(s, wt, wr, chans, snr, ens, seed=seed, variant=variant)
    C_ = chans.shape[1]
    nv, ns = len(wins), len(snr)
    fpc = frames_per_cell(ns, C_, ens)
    out = {}
    for bins, chan in RESOLVE:
        r = handle.ber_run_resolved(s, wt, wr, chans, snr, ens, seed=seed, variant=variant, by_subcarrier=bins, by_channel=chan)
        cr, nr = (C_ if chan else 1), (p.N if bins else 1)
        assert r["bit_err"].shape == r["sym_err"].shape == (nv, ns, cr, nr)
        assert r["sym_tot"].shape == r["bit_tot"].shape == (ns, cr, nr)
        assert np.array_equal(r["sym_err"].sum(axis=(2, 3)), ref["sym_err"]), (bins, chan, r["sym_err"].sum(axis=(2, 3)), ref["sym_err"])
        assert np.array_equal(r["bit_err"].sum(axis=(2, 3)), ref["bit_err"]), (bins, chan)
        assert np.array_equal(r["sym_tot"].sum(axis=(1, 2)), ref["sym_tot"])
        assert np.array_equal(r["bit_tot"], r["sym_tot"] * p.bits)
        cells = fpc if chan else fpc.sum(axis=1, keepdims=True)
        if bins:
            act = p.active
            assert np.array_equal(r["sym_tot"][:, :, act], np.broadcast_to(cells[:, :, None] * (p.S - 1), r["sym_tot"][:, :, act].shape))
            assert not r["sym_tot"][:, :, ~act].any() and not r["sym_err"][..., ~act].any() and not r["bit_err"][..., ~act].any()
        else:
            assert np.array_equal(r["sym_tot"][:, :, 0], cells * int(act_count(p)) * (p.S - 1))
        assert np.all(r["sym_err"] <= r["bit_err"]) and np.all(r["sym_err"] <= r["sym_tot"][None])
        out[(bins, chan)] = r
    both = out[(True, True)]
    assert np.array_equal(both["sym_err"].sum(axis=3), out[(False, True)]["sym_err"][..., 0])
    assert np.array_equal(both["sym_err"].sum(axis=2), out[(True, False)]["sym_err"][:, :, 0, :])
    assert ref["sym_err"].sum() > 0, "a sum identity over zero errors proves nothing"
    return both


def act_count(p):
    return int(np.count_nonzero(p.active))


def kernel_of(handle, s, wins, chans, snr):
    if len(wins) == 1:
        return handle.ber_plan(s, wins[0][0], wins[0][1], chans, snr).kernel
    return handle.ber_plan_multi(s, [w[0] for w in wins], [w[1] for w in wins], chans, snr).kernel


def windows(p, n, seed):
    wins = [O.perturbed_windows(p, seed=seed + k)[:2] for k in range(n - 1)]
    return wins + [(O.rc_window_tx(p), O.rc_window_rx(p))]


# (name, N, cp, tail_tx, tail_rx, bits, L, pairs, precision, no_tconv, kernel check, conv / noise_norm, guard)
CASES = {
    "tconv2_n256": ("WOLA", 256, 16, 8, 10, 4, 21, 1, 0, False, "f32t2_n256", 0, 0),
    "tconv2_n256_7pairs": ("WOLA", 256, 16, 8, 10, 4, 21, 7, 0, False, "f32t2_n256", 0, 0),
    "tconv2_n512": ("CPW", 512, 32, 16, 20, 4, 21, 2, 0, False, "f32t2_n512", 1, 0),
    "tconv2_n1024_cluster": ("WOLA", 1024, 64, 32, 40, 6, 21, 2, 0, False, "f32t2_n1024", 0, 0),
    "tconv2_l84": ("WOLA", 256, 16, 8, 10, 4, 84, 2, 0, False, "_l84", 1, 0),
    "fp64_n256": ("WOLA", 256, 16, 8, 10, 4, 21, 2, 1, False, "f64_n256", 0, 0),
    "circ_n256": ("wrx", 256, 16, 0, 10, 4, 21, 1, 0, True, "_circ", 0, 0),
    "regs_n256": ("WOLA", 256, 16, 8, 10, 4, 21, 1, 0, True, "ber_f32r_n256", 1, 0),
    "regs_n512": ("WOLA", 512, 32, 16, 20, 4, 21, 2, 0, True, "ber_f32r_n512", 0, 0),
    "regs_n1024_cluster": ("WOLA", 1024, 64, 32, 40, 6, 21, 1, 0, True, "_cl2", 1, 0),
    "staged_n64": ("WOLA", 64, 8, 4, 4, 4, 21, 2, 0, False, "_c0_", 0, 0),
    "guard_n256": ("CPW", 256, 22, 8, 10, 4, 21, 2, 0, False, "f32t2_n256", 1, 64),
    "guard_n1024_fp64": ("WOLA", 1024, 64, 32, 40, 6, 21, 1, 1, False, "f64_n1024", 1, 256),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_sum_identity(handle, case, monkeypatch):
    name, N, cp, ttx, trx, bits, L, nv, prec, no_tconv, kern, conv, guard = CASES[case]
    if no_tconv:
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits, noise_norm=conv, constellation=conv, guard=guard)
    s = to_sys(p, prec)
    wins = windows(p, nv, seed=N + cp)
    chans = O.synth_channels(3, L, seed=N + L)
    snr = np.array([4.0, 10.0, 16.0]) + (6.0 if bits == 6 else 0.0)
    k = kernel_of(handle, s, wins, chans, snr)
    assert kern in k, (case, k)
    if no_tconv:
        assert "_c0_" not in k, k                        # a register kernel: the resolved call runs its twin
    check_sum_identity(handle, p, s, wins, chans, snr, 6, seed=N + nv, variant=3)


def cells_vs_oracle(handle, p, precision, L=21):
    """2 SNR points x 3 channels x ensemble 2, every frame replayed through the oracle on the exported draws: fp64 equal
    in every (SNR, channel, bin) cell, fp32 within the cell's boundary-flip budget.  Returns the kernel production runs."""
    s = to_sys(p, precision)
    N = p.N
    vt, vr, _, _ = O.perturbed_windows(p, seed=5)
    chans = O.synth_channels(3, L, seed=9)
    snr = np.array([6.0, 14.0]) + (6.0 if p.bits == 6 else 0.0)
    ens = 2
    k = handle.ber_plan(s, vt, vr, chans, snr).kernel
    r = handle.ber_run_resolved(s, [vt], [vr], chans, snr, ens, seed=21, variant=2, by_subcarrier=True, by_channel=True)
    F = len(snr) * chans.shape[1] * ens
    sym, nz = handle.ber_draws(s, L, 21, 2, np.arange(F))
    want_s = np.zeros((2, 3, N), dtype=np.int64)
    want_b = np.zeros((2, 3, N), dtype=np.int64)
    slack = np.zeros((2, 3, N), dtype=np.int64)
    m, sc = O.qam_levels(p.bits), O.qam_scale(p.bits, p.constellation)
    for f in range(F):
        si, c = f // (3 * ens), (f // ens) % 3
        res = O.frame_chain_structured(p, vt, vr, chans[:, c], snr[si], sym[f].T, nz[f])
        a, b = R.per_bin_errors(p, res, sym[f].T)
        want_s[si, c] += a
        want_b[si, c] += b
        x = res.eq / sc
        near = np.minimum(dist(x.real, m), dist(x.imag, m)) <= 1e-4 * np.maximum(1.0, np.abs(x))
        slack[si, c] += near.sum(axis=1)
    got_s, got_b = r["sym_err"][0], r["bit_err"][0]
    assert want_s.sum() > 0
    if precision == 1:
        assert np.array_equal(got_s, want_s) and np.array_equal(got_b, want_b)
    else:
        assert np.all(np.abs(got_s - want_s) <= slack), (np.abs(got_s - want_s).max(), slack.max())
        assert np.all(np.abs(got_b - want_b) <= 2 * slack)
    return k


@pytest.mark.gpu
@pytest.mark.parametrize("policy,precision", [("tconv2", 0), ("staged", 0), ("staged", 1)])
def test_cells_match_oracle(handle, policy, precision, monkeypatch):
    monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    N = 256 if policy == "tconv2" else 64
    cp, ttx, trx = (16, 8, 10) if N == 256 else (8, 4, 4)
    p = O.system_params("WOLA", N, cp, ttx, trx, S=16, bits=4, noise_norm=1, constellation=1)
    k = cells_vs_oracle(handle, p, precision)
    assert ("f32t2" in k) == (policy == "tconv2") and (precision == 0 or "f64" in k), k


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,cp,ttx,trx,bits,no_tconv,kern", [
    ("WOLA", 256, 16, 8, 10, 4, False, "f32t2_n256"), ("wrx", 256, 16, 0, 10, 4, True, "_circ"),
    ("WOLA", 256, 16, 8, 10, 4, True, "ber_f32r_n256"), ("WOLA", 512, 32, 16, 20, 4, True, "ber_f32r_n512"),
    ("WOLA", 1024, 64, 32, 40, 6, True, "_cl2")])
def test_staged_twin_numbers_noise_like_production(handle, name, N, cp, ttx, trx, bits, no_tconv, kern, monkeypatch):
    """Where the production kernel's own twin cannot hold the accumulators, the staged policy runs with that kernel's noise
    numbering (chunk / split / n48).  Forced here (WOFDM_RESOLVED_STAGED): its cells must match the oracle replayed on the
    draws wofdm_ber_draws exports for the production kernel, within the fp32 boundary-flip budget."""
    monkeypatch.setenv("WOFDM_RESOLVED_STAGED", "1")
    if no_tconv:
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits, noise_norm=0, constellation=0)
    k = cells_vs_oracle(handle, p, 0)
    assert kern in k, k


def dist(v, m):
    b = np.arange(-(m - 2), m - 1, 2.0)
    return np.min(np.abs(v[..., None] - b), axis=-1)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tconv2_n256", "tconv2_n256_fused", "tconv2_n1024_cluster", "staged_n64"])
def test_many_frames_per_cta(handle, case, monkeypatch):
    """The accumulators a CTA carries from frame to frame, flushed when the cell changes.  Long runs: one CTA per SM, 3000
    frames on at most 148 frames in flight, a CTA stays ~3 frames in a cell and crosses several.
    (a) Within the run: by both axes, summed over the bins, equals the by-channel counters, which never touch the
        accumulators (per-warp atomics at the cell's address); summed over the channels it equals the by-sub-carrier run,
        whose cells (SNR points) change at other frames.  An error put into the wrong cell, a lost flush or a missed reset
        breaks one of them.
    (b) Against the same frames as 47 shards of at most 64 frames, where every CTA decides one frame and flushes once
        (draws depend on the frame only): every cell bit for bit."""
    monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    name, N, cp, ttx, trx, bits, nv, kern = {
        "tconv2_n256": ("WOLA", 256, 16, 8, 10, 4, 1, "f32t2_n256"),
        "tconv2_n256_fused": ("WOLA", 256, 16, 8, 10, 4, 3, "f32t2_n256"),
        "tconv2_n1024_cluster": ("WOLA", 1024, 64, 32, 40, 6, 2, "f32t2_n1024"),
        "staged_n64": ("WOLA", 64, 8, 4, 4, 4, 2, "_c0_")}[case]
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits)
    s = to_sys(p, 0)
    wins = windows(p, nv, seed=3)
    wt, wr = [w[0] for w in wins], [w[1] for w in wins]
    chans = O.synth_channels(3, 21, seed=6)
    snr = np.array([4.0, 12.0]) + (6.0 if bits == 6 else 0.0)
    ens, K = 500, 47                                   # 3000 frames; ceil(3000 / 47) = 64 per shard
    assert kern in kernel_of(handle, s, wins, chans, snr)
    run = lambda bins, chan, **kw: handle.ber_run_resolved(s, wt, wr, chans, snr, ens, seed=17, variant=1,
                                                           by_subcarrier=bins, by_channel=chan, **kw)
    monkeypatch.setenv("WOFDM_MAX_CTAS_PER_SM", "1")
    long = {rc: run(*rc) for rc in RESOLVE}
    monkeypatch.delenv("WOFDM_MAX_CTAS_PER_SM")
    both = long[(True, True)]
    assert both["sym_err"].sum() > 0
    for key in ("bit_err", "sym_err"):
        assert np.array_equal(both[key].sum(axis=3), long[(False, True)][key][..., 0]), key
        assert np.array_equal(both[key].sum(axis=2), long[(True, False)][key][:, :, 0, :]), key
    for rc in ((True, False), (True, True)):
        acc = {key: np.zeros_like(long[rc][key]) for key in ("bit_err", "sym_err", "sym_tot")}
        for i in range(K):
            r = run(*rc, shard=(i, K))
            for key in acc:
                acc[key] += r[key]
        for key in acc:
            assert np.array_equal(acc[key], long[rc][key]), (case, rc, key, np.argwhere(acc[key] != long[rc][key])[:5])


@pytest.mark.gpu
def test_shards_add_up(handle):
    p = O.system_params("WOLA", 256, 16, 8, 10, S=16, bits=4)
    s = to_sys(p, 0)
    wins = windows(p, 2, seed=1)
    chans = O.synth_channels(4, 21, seed=2)
    snr = np.array([3.0, 9.0])
    kw = dict(seed=5, by_subcarrier=True, by_channel=True)
    full = handle.ber_run_resolved(s, [w[0] for w in wins], [w[1] for w in wins], chans, snr, 7, **kw)
    parts = [handle.ber_run_resolved(s, [w[0] for w in wins], [w[1] for w in wins], chans, snr, 7, shard=(i, 3), **kw)
             for i in range(3)]
    for key in ("bit_err", "sym_err", "sym_tot"):
        assert np.array_equal(sum(q[key] for q in parts), full[key]), key
    fpc = frames_per_cell(2, 4, 7, (1, 3))
    assert np.array_equal(parts[1]["sym_tot"][:, :, 0], fpc * (p.S - 1))


@pytest.mark.gpu
def test_two_device_handle_matches_one_device(handle):
    n = C.c_int(0)
    assert W.capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("one visible device")
    p = O.system_params("WOLA", 256, 16, 8, 10, S=16, bits=4)
    s = to_sys(p, 0)
    vt, vr, _, _ = O.perturbed_windows(p, seed=1)
    chans = O.synth_channels(3, 21, seed=2)
    one = handle.ber_run_resolved(s, [vt], [vr], chans, [4.0, 8.0], 9, seed=3, by_channel=True)
    with W.Handle([0, 1]) as h2:
        two = h2.ber_run_resolved(s, [vt], [vr], chans, [4.0, 8.0], 9, seed=3, by_channel=True)
    for key in ("bit_err", "sym_err", "sym_tot"):
        assert np.array_equal(one[key], two[key]), key


@pytest.mark.gpu
def test_errors_and_handle_survives(handle):
    p = O.system_params("WOLA", 64, 8, 4, 4, S=4, bits=4)
    s = to_sys(p, 0)
    vt, vr, _, _ = O.perturbed_windows(p, seed=1)
    chans = O.synth_channels(2, 5, seed=2)
    lib = W.capi.load()
    wt, wr = np.ascontiguousarray(vt, dtype=np.float64), np.ascontiguousarray(vr, dtype=np.float64)
    ch = np.ascontiguousarray(np.stack([chans.real.T, chans.imag.T], axis=-1), dtype=np.float64)
    snr = np.array([5.0])
    out = [np.zeros(2 * 64, dtype=np.int64) for _ in range(3)]
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))

    def call(resolve, ptrs):
        return lib.wofdm_ber_run_resolved(handle._h, C.byref(s), dp(wt), dp(wr), 1, dp(ch), 5, 2, dp(snr), 1, 2, 0, 0, 0, 1,
                                          resolve, *ptrs)
    for resolve in (0, 4, 5, -1):
        assert call(resolve, [ip(o) for o in out]) == W.capi.EINVAL
    for k in range(3):
        ptrs = [ip(o) for o in out]
        ptrs[k] = None
        assert call(1, ptrs) == W.capi.EINVAL
    assert call(3, [ip(o) for o in out]) == W.capi.OK
    r = handle.ber_run_resolved(s, [vt], [vr], chans, snr, 2, by_channel=True)
    ref = handle.ber_run(s, vt, vr, chans, snr, 2)
    assert np.array_equal(r["sym_err"].sum(axis=(2, 3))[0], ref["sym_err"])


@pytest.mark.gpu
def test_wofdm_system_mirror(handle, tmp_path):
    """run_simulation_per_subcarrier averaged over the active bins is run_simulation's SER, for the same seed."""
    from wofdm_b200 import ofdm_utils as U
    chans = O.synth_channels(3, 21, seed=4)
    snr = np.array([2.0, 8.0, 14.0])
    for name, cp, ttx, trx in (("WOLA", 16, 8, 10), ("CP", 16, 0, 0)):
        sysm = U.wOFDMSystem(name, 256, cp, ttx, trx, str(tmp_path), seed=11, handle=handle)
        p = O.system_params(name, 256, cp, ttx, trx, S=16)
        vt, vr, _, _ = O.perturbed_windows(p, seed=2)
        ref = sysm.run_simulation(chans, np.diag(vt), np.diag(vr), 5, snr, 16)
        per = sysm.run_simulation_per_subcarrier(chans, np.diag(vt), np.diag(vr), 5, snr, 16)
        if name == "CP":
            ref, per = (ref,), (per,)
        for a, b in zip(ref, per):
            assert b.shape == (3, 256)
            np.testing.assert_allclose(b.mean(axis=1), a, rtol=1e-12, atol=0)
