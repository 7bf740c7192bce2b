"""Several window pairs and roll-offs of the channel-mask chain on the same frames in one call (wofdm_ber_run_masked_multi,
Handle.ber_run_masked_multi, ofdm_utils.run_sim_mc_multi).

GPU: pair v's counters equal ber_run_masked with pair v's windows, roll-off and variant + v, bit for bit, on every path the
masked chain takes (the gathering tensor-core kernel for all pairs in one launch, one launch per pair on the assembled
stream, the staged kernel, the per-symbol FFT mask), across product batches, shards and devices; one pair is the single
call; the refusals leave the handle usable.  CPU: the mirror's argument handling.
"""
import ctypes as C

import numpy as np
import pytest

import wofdm_b200 as W
from oracle import wofdm_oracle as O

ENV = ("WOFDM_DEBUG", "WOFDM_MASK_FFT", "WOFDM_MASK_DUMP", "WOFDM_RESOLVED_STAGED", "WOFDM_NO_TCONV", "WOFDM_VARIANT")
ROLL_OFFS = [4, 10, 30, 6, 14, 20, 40, 8]


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


def pairs(p, s, n_var):
    """pair 0: the RC windows; pair v > 0: RC perturbed by a seeded +-10 % (Tx and Rx)"""
    wt, wr = [W.capi.rc_window_tx(s)], [W.capi.rc_window_rx(s)]
    for v in range(1, n_var):
        vt, vr, _, _ = O.perturbed_windows(p, seed=100 + v)
        wt.append(vt)
        wr.append(vr)
    return np.array(wt), np.array(wr), ROLL_OFFS[:n_var]


def check_against_singles(handle, s, wt, wr, ro, chans, snr, ens, seed=5, variant=3, shard=(0, 1)):
    m = handle.ber_run_masked_multi(s, wt, wr, chans, snr, ens, seed=seed, variant=variant, roll_offs=ro, shard=shard)
    n_var = len(ro)
    assert m["bit_err"].shape == m["sym_err"].shape == (n_var, len(snr))
    for v in range(n_var):
        r = handle.ber_run_masked(s, wt[v], wr[v], chans, snr, ens, seed=seed, variant=variant + v, roll_off=ro[v], shard=shard)
        assert np.array_equal(m["bit_err"][v], r["bit_err"]), (v, m["bit_err"][v], r["bit_err"])
        assert np.array_equal(m["sym_err"][v], r["sym_err"]), (v, m["sym_err"][v], r["sym_err"])
        assert np.array_equal(m["bit_tot"], r["bit_tot"]) and np.array_equal(m["sym_tot"], r["sym_tot"])
    if n_var > 1:       # a mix-up of pairs cannot pass
        assert len({tuple(row) for row in m["bit_err"]}) == n_var, m["bit_err"]
        assert np.all(m["bit_err"].sum(axis=1) > 0), m["bit_err"]
    return m


# (system, N, cp, tail_tx, tail_rx, bits, S, L, guard, n_var)
CASES = {
    "gather_n256_v1": ("wtx", 256, 16, 8, 0, 4, 16, 21, 64, 1),
    "gather_n256_v2": ("wtx", 256, 16, 8, 0, 4, 16, 21, 64, 2),
    "gather_n256_v8": ("wtx", 256, 16, 8, 0, 4, 16, 21, 64, 8),
    "gather_n512": ("CPW", 512, 32, 16, 20, 4, 16, 21, 128, 3),
    "staged_n128": ("CP", 128, 8, 0, 0, 2, 16, 21, 16, 3),
    "stream_s4": ("WOLA", 256, 30, 8, 10, 4, 4, 21, 64, 3),
    "assembled_l40": ("wtx", 256, 16, 8, 0, 4, 16, 40, 64, 3),
    "guard0": ("WOLA", 256, 22, 8, 10, 4, 16, 21, 0, 3),
    "wide_guard": ("wtx", 256, 16, 8, 0, 4, 16, 21, 100, 3),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_pairs_equal_single_calls(handle, case, clean_env):
    name, N, cp, ttx, trx, bits, S, L, guard, n_var = CASES[case]
    p = O.system_params(name, N, cp, ttx, trx, S=S, bits=bits, noise_norm=1, constellation=1, guard=guard)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, n_var)
    chans = O.synth_channels(3, L, seed=N + L)
    check_against_singles(handle, s, wt, wr, ro, chans, [6.0, 14.0], 40)


@pytest.mark.gpu
def test_more_than_one_batch_and_shards(handle, clean_env):
    """17 000 frames (more than the product's batch of 16 384); shards 1 and 3 each against the single calls, and the three
    shards add up to the whole job."""
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 3)
    chans = O.synth_channels(5, 21, seed=6)
    snr, ens = [4.0, 10.0], 1700
    full = check_against_singles(handle, s, wt, wr, ro, chans, snr, ens)
    acc = {k: np.zeros_like(v) for k, v in full.items()}
    for k in range(3):
        part = check_against_singles(handle, s, wt, wr, ro, chans, snr, ens, shard=(k, 3))
        for key in acc:
            acc[key] += part[key]
    for key in acc:
        assert np.array_equal(acc[key], full[key]), key


@pytest.mark.gpu
def test_mask_fft_path(handle, clean_env):
    clean_env.setenv("WOFDM_MASK_FFT", "1")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 3)
    check_against_singles(handle, s, wt, wr, ro, O.synth_channels(2, 21, seed=9), [6.0, 14.0], 30)


@pytest.mark.gpu
def test_two_device_handle_matches_one_device(handle, clean_env):
    n = C.c_int(0)
    assert W.capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("one visible device")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 3)
    chans = O.synth_channels(3, 21, seed=2)
    one = handle.ber_run_masked_multi(s, wt, wr, chans, [4.0, 8.0], 300, seed=3, variant=1, roll_offs=ro)
    with W.Handle([0, 1]) as h2:
        two = h2.ber_run_masked_multi(s, wt, wr, chans, [4.0, 8.0], 300, seed=3, variant=1, roll_offs=ro)
    for key in one:
        assert np.array_equal(one[key], two[key]), key


@pytest.mark.gpu
def test_one_pair_is_the_single_call(handle, clean_env):
    from wofdm_b200 import ofdm_utils as U
    p = O.system_params("WOLA", 256, 22, 8, 10, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    vt, vr, _, _ = O.perturbed_windows(p, seed=7)
    chans = O.synth_channels(2, 21, seed=7)
    m = handle.ber_run_masked_multi(s, [vt], [vr], chans, [8.0], 50, seed=2, variant=4, roll_offs=14)
    r = handle.ber_run_masked(s, vt, vr, chans, [8.0], 50, seed=2, variant=4, roll_off=14)
    for key in r:
        assert np.array_equal(m[key].reshape(r[key].shape), r[key]), key
    args = (7, p.cp, p.cs, 8, 10, np.diag(vt), np.diag(vr), chans[:, 0], 12.0, 64, p.rm, p.shift, 256, 4, 16)
    bm, b0 = U.run_sim_mc(*args, 10, seed=3, handle=handle)
    mm, m0 = U.run_sim_mc_multi(*args[:5], [args[5]], [args[6]], *args[7:], [10], seed=3, handle=handle)
    assert mm.shape == m0.shape == (1,)
    assert mm[0] == bm and m0[0] == b0
    # two configurations: configuration v is run_sim_mc's chain with unmasked noise stream v and masked stream 2 + v
    vt2, vr2, _, _ = O.perturbed_windows(p, seed=8)
    mm, m0 = U.run_sim_mc_multi(*args[:5], [vt, vt2], [vr, vr2], *args[7:], [10, 30], seed=3, handle=handle)
    s0 = to_sys(p)
    r1 = handle.ber_run_masked(s0, vt2, vr2, chans[:, :1], [12.0], 7, seed=3, variant=3, roll_off=30)
    u1 = handle.ber_run(s0, vt2, vr2, chans[:, :1], [12.0], 7, seed=3, variant=1)
    assert mm[1] == r1["bit_err"][0] / r1["bit_tot"][0] and m0[1] == u1["bit_err"][0] / u1["bit_tot"][0]


@pytest.mark.gpu
def test_refusals_and_handle_survives(handle, clean_env):
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, _ = pairs(p, s, 8)
    chans = O.synth_channels(2, 21, seed=2)
    lib = W.capi.load()
    ch = np.ascontiguousarray(chans.T, dtype=np.complex128)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    rp = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))
    snr = np.array([6.0])
    out = [np.zeros(8, dtype=np.int64) for _ in range(4)]

    def call(n_var, ro, sys=s, wt_=wt, wr_=wr):
        roa = None if ro is None else np.ascontiguousarray(ro, dtype=np.int32)
        return lib.wofdm_ber_run_masked_multi(handle._h, C.byref(sys), dp(wt_), dp(wr_), None if roa is None else rp(roa), n_var,
                                              dp(ch), 21, 2, dp(snr), 1, 4, 0, 0, 0, 1, ip(out[0]), ip(out[1]), ip(out[2]),
                                              ip(out[3]))

    ref = handle.ber_run_masked_multi(s, wt[:2], wr[:2], chans, snr, 4, roll_offs=[4, 10])

    def still_works():
        r = handle.ber_run_masked_multi(s, wt[:2], wr[:2], chans, snr, 4, roll_offs=[4, 10])
        for key in ref:
            assert np.array_equal(r[key], ref[key]), key

    ok = [4, 10, 30, 6, 14, 20, 40, 8]
    assert call(8, ok) == W.capi.OK
    for n_var in (0, 9):
        assert call(n_var, ok + [4]) == W.capi.EINVAL
    assert call(4, None) == W.capi.EINVAL
    bad = list(ok)
    bad[3] = 10 ** 4                        # pair 3 only: a roll-off the mask cannot hold
    assert call(8, bad) == W.capi.EINVAL
    bad[3] = 0
    assert call(8, bad) == W.capi.EINVAL
    still_works()
    assert call(2, ok, sys=s.copy(precision=1)) == W.capi.EUNSUPPORTED
    p1k = O.system_params("wtx", 1024, 64, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s1k = to_sys(p1k)
    assert call(2, ok, sys=s1k, wt_=np.ones((2, s1k.n_tx)), wr_=np.ones((2, 1024))) == W.capi.EUNSUPPORTED
    still_works()


def test_mirror_argument_handling(monkeypatch):
    """run_sim_mc_multi and Handle.ber_run_masked_multi check their lists before any device work: mismatched lengths are
    refused, a scalar roll-off is broadcast to every pair."""
    from wofdm_b200 import ofdm_utils as U
    args = (7, 16, 16, 8, 0)
    tail = (np.zeros(21), 12.0, 64, 0, 0, 256, 4, 16)
    wt, wr = np.ones(288), np.ones(256)
    for wts, wrs, ros in (([wt, wt], [wr], [10, 10]), ([wt], [wr], [10, 20]), ([wt, wt], [wr, wr], [10]), ([], [], [])):
        with pytest.raises(ValueError):
            U.run_sim_mc_multi(*args, wts, wrs, *tail, ros, handle=object())
    assert np.array_equal(W.capi._roll_offs(10, 3), [10, 10, 10])
    assert W.capi._roll_offs([4, 10], 2).dtype == np.int32
    for bad in ([4, 10], [[4, 10, 30]], 10.5):
        with pytest.raises(W.WofdmError):
            W.capi._roll_offs(bad, 3)
