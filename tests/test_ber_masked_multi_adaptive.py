"""The channel-mask chain's stopping rule for several window pairs and roll-offs on the same frames in one call
(wofdm_ber_run_masked_adaptive_multi, Handle.ber_run_masked_adaptive_multi, ofdm_utils.run_sim_mc_multi_adaptive).

GPU: the schedule of oracle/adaptive.py over 2 n_var rows (block 0 the masked chain of pair v on noise stream
variant + n_var + v, block 1 its unmasked chain on variant + v), fed by per-ensemble-index counters from one-index segments
of the two chains, for bit and symbol targets; one pair is ber_run_masked_adaptive; an unreachable target is the fixed run;
two shards in two threads with a summing reduce give the one-process result; refusals leave the handle usable.
CPU: the mirror's argument handling and shapes.
"""
import ctypes as C
import threading

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import ofdm_utils as U
from oracle import adaptive as A
from oracle import wofdm_oracle as O
from test_ber_masked_multi import clean_env, pairs, to_sys  # noqa: F401 -- clean_env is a fixture


@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def mask_job(n_var):
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, n_var)
    return p, s, wt, wr, ro, O.synth_channels(4, 21, seed=5), np.array([0.0, 6.0, 12.0, 18.0])


def target_kw(kind, target):
    return {"target_bit_errors": target} if kind == A.BIT else {"target_symbol_errors": target}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [A.SYM, A.BIT])
def test_schedule_matches_oracle(handle, kind, clean_env):
    """Per-(point, e) counts of the 2 n_var rows from one-index segments of both chains, fed to oracle/adaptive.py: the
    adaptive call returns its ensemble_used, counters and rounds exactly, with targets that stop the points in different
    rounds."""
    n_var, E, seed, variant = 3, 16, 9, 2
    p, s, wt, wr, ro, chans, snr = mask_job(n_var)
    bit = np.zeros((2, n_var, 4, E), dtype=np.int64)
    sym = np.zeros((2, n_var, 4, E), dtype=np.int64)
    for e in range(E):
        one_idx = [(k, e, 1) for k in range(4)]
        rm = handle.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, one_idx, seed=seed, variant=variant + n_var,
                                                  roll_offs=ro)
        ru = handle.ber_run_segments(s, wt, wr, chans, snr, E, one_idx, seed=seed, variant=variant)
        bit[0, :, :, e], sym[0, :, :, e] = rm["bit_err"], rm["sym_err"]
        bit[1, :, :, e], sym[1, :, :, e] = ru["bit_err"], ru["sym_err"]
    rows_b, rows_s = bit.reshape(2 * n_var, 4, E), sym.reshape(2 * n_var, 4, E)
    m_all = (rows_b if kind == A.BIT else rows_s).sum(axis=2).min(axis=0)
    assert m_all.min() > 0
    tested = set()
    for target in sorted({int(x) for x in np.geomspace(max(1, m_all.min() // 8), m_all.max(), 7)}):
        used, tb, ts, rounds, blocks = A.schedule(rows_b, rows_s, target, kind, first_block=1)
        stop_round = [max(i for i, rnd in enumerate(blocks) if k in rnd) for k in range(4)]
        r = handle.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, E, first_block=1, seed=seed, variant=variant,
                                                 roll_offs=ro, **target_kw(kind, target))
        assert r["bit_err"].shape == r["sym_err"].shape == (2, n_var, 4)
        assert r["ensemble_used"].tolist() == used, (target, r["ensemble_used"], used)
        assert r["bit_err"].reshape(2 * n_var, 4).tolist() == tb, target
        assert r["sym_err"].reshape(2 * n_var, 4).tolist() == ts and r["rounds"] == rounds, target
        assert np.array_equal(r["sym_tot"], np.asarray(used) * chans.shape[1] * int(p.active.sum()) * (p.S - 1))
        tested.add(len(set(stop_round)))
    assert max(tested) >= 3, "the targets must stop points in different rounds"


@pytest.mark.gpu
def test_one_pair_is_the_single_call(handle, clean_env):
    p, s, wt, wr, ro, chans, snr = mask_job(1)
    for kw in (dict(target_bit_errors=300), dict(target_symbol_errors=200, first_block=2)):
        m = handle.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, 30, seed=4, variant=5, roll_offs=ro, **kw)
        r = handle.ber_run_masked_adaptive(s, wt[0], wr[0], chans, snr, 30, seed=4, variant=5, roll_off=ro[0], **kw)
        for key in ("bit_err", "sym_err"):
            assert np.array_equal(m[key][:, 0], r[key]), key
        for key in ("bit_tot", "sym_tot", "ensemble_used", "rounds"):
            assert np.array_equal(m[key], r[key]), key
        assert m["ensemble_used"].min() < 30


@pytest.mark.gpu
def test_unreachable_target_is_the_fixed_run(handle, clean_env):
    """Block 0 is ber_run_masked_multi(ensemble_max, variant + n_var) and block 1 ber_run_multi(ensemble_max, variant)."""
    n_var, E, seed, variant = 4, 6, 7, 2
    p, s, wt, wr, ro, chans, snr = mask_job(n_var)
    masked = handle.ber_run_masked_multi(s, wt, wr, chans, snr, E, seed=seed, variant=variant + n_var, roll_offs=ro)
    plain = handle.ber_run_multi(s, wt, wr, chans, snr, E, seed=seed, variant=variant)
    for kw in (dict(target_symbol_errors=10 ** 15), dict(target_bit_errors=10 ** 15, first_block=E)):
        r = handle.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, E, seed=seed, variant=variant, roll_offs=ro, **kw)
        assert np.array_equal(r["ensemble_used"], np.full(len(snr), E))
        assert r["rounds"] == (1 if "first_block" in kw else 3)
        for block, ref in enumerate((masked, plain)):
            assert np.array_equal(r["bit_err"][block], ref["bit_err"]), block
            assert np.array_equal(r["sym_err"][block], ref["sym_err"]), block
            assert np.array_equal(r["bit_tot"], ref["bit_tot"]) and np.array_equal(r["sym_tot"], ref["sym_tot"])
    assert len({tuple(row) for row in masked["bit_err"]}) == n_var


@pytest.mark.gpu
def test_shards_in_two_threads(clean_env):
    """Two handles on device 0, shards (0, 2) and (1, 2), summed by a threading.Barrier reducer on counts of shape
    (2, n_var, n_snr, 2): each returns the single-process result."""
    n_var = 3
    p, s, wt, wr, ro, chans, snr = mask_job(n_var)
    with W.Handle([0]) as h0:
        first = h0.ber_run_masked_segments(s, wt[0], wr[0], chans, snr, 40, [(k, 0, 1) for k in range(len(snr))], seed=3,
                                           variant=n_var, roll_off=ro[0])
        kw = dict(target_symbol_errors=4 * int(first["sym_err"].max()) + 1, first_block=1, seed=3, roll_offs=ro)
        want = h0.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, 40, **kw)
    bar = threading.Barrier(2, timeout=300)
    slots, out = [None, None], [None, None]

    def reducer(rank):
        def red(counts):
            assert counts.shape == (2, n_var, len(snr), 2)
            slots[rank] = counts.copy()
            bar.wait()
            tot = slots[0] + slots[1]
            bar.wait()
            return tot
        return red

    def run(rank):
        with W.Handle([0]) as h:
            out[rank] = h.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, 40, shard=(rank, 2), reduce=reducer(rank), **kw)
    th = [threading.Thread(target=run, args=(r,)) for r in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join(timeout=600)
    assert want["ensemble_used"].min() < 40 and want["rounds"] >= 2
    for r in out:
        assert r is not None
        for key in ("bit_err", "sym_err", "bit_tot", "sym_tot", "ensemble_used", "rounds"):
            assert np.array_equal(r[key], want[key]), key


def _raw(handle, s, wt, wr, chans, ro, n_var):
    wt, wr = np.ascontiguousarray(wt, dtype=np.float64), np.ascontiguousarray(wr, dtype=np.float64)
    chf = np.ascontiguousarray(np.asarray(chans, dtype=np.complex128).T)
    L, Cn = chans.shape
    snr = np.array([6.0, 12.0])
    o = [np.zeros(64, dtype=np.int64) for _ in range(5)]
    rounds = C.c_int(0)
    rop = None if ro is None else np.ascontiguousarray(ro, dtype=np.int32).ctypes.data_as(C.POINTER(C.c_int))
    return W.capi.load().wofdm_ber_run_masked_adaptive_multi(
        handle._h, C.byref(s), wt.ctypes.data_as(W.capi._dp), wr.ctypes.data_as(W.capi._dp), rop, n_var,
        chf.ctypes.data_as(W.capi._dp), L, Cn, snr.ctypes.data_as(W.capi._dp), 2, 8, 1, W.capi.WOFDM_TARGET_BIT_ERRORS, 100,
        1, 0, 0, 1, W.capi.REDUCE_FN(), None, *[x.ctypes.data_as(W.capi._i64p) for x in o], C.byref(rounds))


@pytest.mark.gpu
def test_refusals_leave_the_handle_usable(handle, clean_env):
    p, s, wt, wr, ro, chans, snr = mask_job(8)
    wt9, wr9 = np.vstack([wt, wt[:1]]), np.vstack([wr, wr[:1]])
    want = handle.ber_run_masked_adaptive_multi(s, wt[:2], wr[:2], chans, snr, 8, target_bit_errors=100, seed=1,
                                                roll_offs=ro[:2])
    for kw in (dict(n_var=0), dict(wt=wt9, wr=wr9, ro=list(ro) + [4], n_var=9), dict(ro=None), dict(ro=[4, 1000])):
        args = dict(wt=wt[:2], wr=wr[:2], ro=ro[:2], n_var=2)
        args.update(kw)
        assert _raw(handle, s, args["wt"], args["wr"], chans, args["ro"], args["n_var"]) == W.capi.EINVAL, kw
        again = handle.ber_run_masked_adaptive_multi(s, wt[:2], wr[:2], chans, snr, 8, target_bit_errors=100, seed=1,
                                                     roll_offs=ro[:2])
        for key in want:
            assert np.array_equal(again[key], want[key]), (kw, key)


@pytest.mark.gpu
def test_two_device_handle_matches_one_device(handle, clean_env):
    n = C.c_int(0)
    assert W.capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("needs two GPUs")
    p, s, wt, wr, ro, chans, snr = mask_job(3)
    kw = dict(target_bit_errors=2000, seed=6, roll_offs=ro)
    one = handle.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, 400, **kw)
    with W.Handle([0, 1]) as h2:
        two = h2.ber_run_masked_adaptive_multi(s, wt, wr, chans, snr, 400, **kw)
    for key in one:
        assert np.array_equal(one[key], two[key]), key


def mc_args(n_var, N=256):
    """the positional arguments of run_sim_mc_multi_adaptive up to rollOff, with n_var RC window pairs"""
    p = O.system_params("wtx", N, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    wt, wr = O.rc_window_tx(p), O.rc_window_rx(p)
    return [5, p.cp, p.cs, p.tail_tx, p.tail_rx, [np.diag(wt)] * n_var, [np.diag(wr)] * n_var, O.synth_channels(2, 21, 3).T,
            [4.0, 10.0], p.guard, p.rm, p.shift, p.N, p.bits, p.S]


@pytest.mark.gpu
def test_run_sim_mc_multi_adaptive_mirror(handle, clean_env):
    """One configuration equals run_sim_mc_adaptive exactly; three give (n_var, n_snr) rates and the ensemble used."""
    a = mc_args(1)
    single = U.run_sim_mc_adaptive(*a[:5], a[5][0], a[6][0], *a[7:], 10, 200, seed=2, handle=handle)
    multi = U.run_sim_mc_multi_adaptive(*a, [10], 200, seed=2, handle=handle)
    for x, y in zip(multi, single):
        assert np.array_equal(np.squeeze(x), y)
    a = mc_args(3)
    bm, b, used = U.run_sim_mc_multi_adaptive(*a, [4, 10, 30], 200, seed=2, handle=handle)
    assert bm.shape == b.shape == (3, 2) and used.shape == (2,)
    assert np.all(used >= 1) and np.all(used <= 5)


class _Recorder:
    """a stand-in Handle that records the call and returns zero counts of the library's shapes"""
    def __init__(self):
        self.calls = []

    def ber_run_masked_adaptive_multi(self, s, wts, wrs, ch, snr, ensemble_max, **kw):
        self.calls.append((s, wts, wrs, ch, snr, ensemble_max, kw))
        n = len(snr)
        z = np.ones((2, len(wts), n), dtype=np.int64)
        return dict(bit_err=z, sym_err=z, bit_tot=np.full(n, 4), sym_tot=np.full(n, 1), ensemble_used=np.full(n, 3))

    def psd_masked_multi(self, s, wts, roll_offs, frames, seed, estimator):
        self.calls.append((s, wts, roll_offs, frames, seed, estimator))
        x = np.ones((len(wts), 8 * s.N))
        return x, 2 * x


def test_mirrors_argument_handling():
    rec = _Recorder()
    a = mc_args(3)
    bm, b, used = U.run_sim_mc_multi_adaptive(*a, 12, 77, seed=4, handle=rec)
    s, wts, wrs, ch, snr, ens, kw = rec.calls[-1]
    assert kw["roll_offs"] == [12, 12, 12] and kw["target_bit_errors"] == 77 and kw["variant"] == 0 and kw["seed"] == 4
    assert len(wts) == len(wrs) == 3 and ch.shape == (21, 2) and ens == 5
    assert bm.shape == b.shape == (3, 2) and used.shape == (2,)
    U.run_sim_mc_multi_adaptive(*a, [4, 10, 30], 77, handle=rec)
    assert rec.calls[-1][-1]["roll_offs"] == [4, 10, 30]
    with pytest.raises(ValueError):
        U.run_sim_mc_multi_adaptive(*a, [4, 10], 77, handle=rec)
    bad = list(a)
    bad[6] = bad[6][:2]
    with pytest.raises(ValueError):
        U.run_sim_mc_multi_adaptive(*bad, 10, 77, handle=rec)
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    w = [np.diag(O.rc_window_tx(p))] * 2
    r = U.psd_sim_mc_multi(8, p.cp, p.cs, p.tail_tx, w, p.guard, p.N, p.bits, p.S, 10, seed=3, handle=rec)
    assert rec.calls[-1][2] == [10, 10]
    assert r["X_est_masked"].shape == r["X_est"].shape == (2, 2048)
    assert r["obr_masked"].shape == r["obr"].shape == (2,) and np.allclose(r["obr"], 2.0)
    assert r["mf_band_masked"].shape == r["mf_band"].shape == (2, 2048 - 2 * 512) and r["f_axis"].shape == (2048,)
    with pytest.raises(ValueError):
        U.psd_sim_mc_multi(8, p.cp, p.cs, p.tail_tx, w, p.guard, p.N, p.bits, p.S, [4, 10, 30], handle=rec)
    with pytest.raises(ValueError):
        U.psd_sim_mc_multi(8, p.cp, p.cs, p.tail_tx, [], p.guard, p.N, p.bits, p.S, 10, handle=rec)
    with pytest.raises(ValueError):
        U.psd_sim_mc_multi(8, p.cp, p.cs, p.tail_tx, w, 0, p.N, p.bits, p.S, 10, handle=rec)


def test_handle_checks_roll_offs_before_the_call():
    """Handle.psd_masked_multi / ber_run_masked_*_multi refuse a roll-off list of the wrong length before any device work."""
    h = W.Handle.__new__(W.Handle)          # (no device needed: the checks run before the library is called)
    h._h = None
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    w = np.array([O.rc_window_tx(p)] * 2)
    with pytest.raises(W.capi.WofdmError):
        h.psd_masked_multi(s, w, roll_offs=[4, 10, 30])
    with pytest.raises(W.capi.WofdmError):
        h.psd_masked_multi(s, w[:, :-1], roll_offs=10)
