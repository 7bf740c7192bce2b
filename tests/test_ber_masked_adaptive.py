"""Frame segments and the stopping rule of the channel-mask chain (wofdm_ber_run_masked_segments,
wofdm_ber_run_masked_adaptive).

CPU: the masked chain's shard rule of sharding.segment_frame_ids.
GPU: on every kernel row of test_ber_masked_resolved.CASES, segment lists add up to wofdm_ber_run_masked and, cell by cell,
to wofdm_ber_run_masked_resolved, through the twin of the kernel the fixed call runs; shards of a list larger than one mask
batch add up exactly; replayed draws agree with the oracle's masked chain; an unreachable target is the two fixed calls of
run_sim_mc; the schedule equals oracle/adaptive.py on measured per-index counts of both chains; shards in two threads; error
codes; the run_sim_mc mirror.
"""
import ctypes as C
import re
import threading

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import sharding
from oracle import adaptive as A
from oracle import ber_resolved as R
from oracle import wofdm_oracle as O
from test_ber_masked_resolved import (CASES, case_setup, check_cells_and_totals, clean_env, dist, kernels_of,  # noqa: F401
                                      one, to_sys)


# ---------------------------------------------------------------- CPU

def test_segment_frame_ids_contiguous_shards():
    segs = [(1, 2, 2), (0, 0, 1)]
    f = sharding.segment_frame_ids(segs, 3, 5)
    assert f.tolist() == [17, 18, 22, 23, 27, 28, 0, 5, 10]
    parts = [sharding.segment_frame_ids(segs, 3, 5, shard=(k, 4), contiguous=True) for k in range(4)]
    assert [p.tolist() for p in parts] == [[17, 18], [22, 23], [27, 28], [0, 5, 10]]     # [floor(9k/4), floor(9(k+1)/4))
    assert np.array_equal(np.concatenate(parts), f)
    assert sharding.segment_frame_ids(segs, 3, 5, shard=(0, 1), contiguous=True).tolist() == f.tolist()


# ---------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


# every point in interleaved, out-of-order pieces, some of one ensemble index; together [0, 5) of each of the 3 points
SEGS = [(2, 2, 3), (0, 0, 2), (1, 4, 1), (1, 2, 2), (2, 0, 2), (0, 2, 3), (1, 0, 1), (1, 1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_segments_add_up(handle, case, clean_env, capfd):
    """resolve 0 equals ber_run_masked(ensemble_max) bit for bit; two disjoint lists resolved by sub-carrier and channel add
    up to ber_run_masked_resolved(ensemble_max) cell by cell; every segment call runs the twin of the fixed call's kernel
    (WOFDM_MASK_FFT=1: the segmented tx_mask_kernel feeds it)."""
    p, s, vt, vr, L, fft, kp, kt = case_setup(case)
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    chans = O.synth_channels(3, L, seed=p.N + L)
    snr = np.array([6.0, 12.0, 18.0]) + (0.0 if p.bits > 2 else -6.0)
    E = 5
    kw = dict(seed=p.N + p.cp, variant=1, roll_off=10)
    ref, kref = kernels_of(lambda: handle.ber_run_masked(s, vt, vr, chans, snr, E, **kw), clean_env, capfd)
    assert re.fullmatch(kp, one(kref)), (case, kref)
    assert ref["sym_err"].sum() > 0
    r, kseg = kernels_of(lambda: handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, SEGS, **kw), clean_env, capfd)
    assert re.fullmatch(kt, one(kseg)), (case, kseg)
    for key in ("bit_err", "sym_err", "sym_tot", "bit_tot"):
        assert np.array_equal(r[key], ref[key]), (case, key, r[key], ref[key])
    full = handle.ber_run_masked_resolved(s, vt, vr, chans, snr, E, by_subcarrier=True, by_channel=True, **kw)
    a = handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, SEGS[:3], by_subcarrier=True, by_channel=True, **kw)
    b = handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, SEGS[3:], by_subcarrier=True, by_channel=True, **kw)
    for key in ("bit_err", "sym_err", "sym_tot", "bit_tot"):
        assert a[key].shape == full[key].shape == (3, 3, p.N)
        assert np.array_equal(a[key] + b[key], full[key]), (case, key)


@pytest.mark.gpu
@pytest.mark.parametrize("fft", [False, True])
def test_shards_add_up(handle, fft, clean_env):
    """A segment list of 17 000 frames, more than one batch of the mask product (16 384; 8 192 for the FFT kernel): 1, 2, 3
    and 47 shards add up to ber_run_masked with no tolerance, and each shard's sym_tot counts the frames the contiguous
    rule gives it."""
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    vt, vr, _, _ = O.perturbed_windows(p, seed=3)
    Cn, E = 5, 1700
    chans = O.synth_channels(Cn, 21, seed=6)
    snr = np.array([4.0, 10.0])
    kw = dict(seed=17, variant=1, roll_off=10)
    segs = [(1, 0, 900), (0, 800, 900), (1, 900, 800), (0, 0, 800)]
    full = handle.ber_run_masked(s, vt, vr, chans, snr, E, **kw)
    assert full["sym_err"].sum() > 10 ** 5
    per_frame = int(p.active.sum()) * (p.S - 1)
    for W_ in (1, 2, 3, 47):
        acc = {key: np.zeros_like(full[key]) for key in full}
        for k in range(W_):
            part = handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, segs, shard=(k, W_), **kw)
            ids = sharding.segment_frame_ids(segs, Cn, E, shard=(k, W_), contiguous=True)
            si, _, _ = sharding.decode(ids, Cn, E)
            assert np.array_equal(part["sym_tot"], np.bincount(si, minlength=2) * per_frame), (W_, k)
            for key in acc:
                acc[key] += part[key]
        for key in acc:
            assert np.array_equal(acc[key], full[key]), (W_, key, acc[key], full[key])


@pytest.mark.gpu
@pytest.mark.parametrize("fft", [False, True])
def test_replay_through_oracle(handle, fft, clean_env):
    """The frames of one shard of a small segment job, exported with segment_frame_ids(contiguous=True) and ber_draws and
    replayed through the oracle's masked chain: every (SNR, channel, bin) cell within the boundary-flip slack of
    test_ber_masked_resolved.test_cells_match_oracle."""
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    L, Cn, E, seed, variant = 21, 3, 4, 23, 1
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    vt, vr, _, _ = O.perturbed_windows(p, seed=5)
    chans = O.synth_channels(Cn, L, seed=9)
    snr = np.array([8.0, 16.0])
    segs, shard = [(1, 1, 2), (0, 3, 1), (0, 0, 2)], (1, 2)
    r = handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, segs, seed=seed, variant=variant, roll_off=10, shard=shard,
                                       by_subcarrier=True, by_channel=True)
    ids = sharding.segment_frame_ids(segs, Cn, E, shard=shard, contiguous=True)
    si, ci, _ = sharding.decode(ids, Cn, E)
    sym, nz = handle.ber_draws(s, L, seed, variant, ids)
    want_s, want_b, slack = (np.zeros((2, Cn, p.N), dtype=np.int64) for _ in range(3))
    m, sc = O.qam_levels(p.bits), O.qam_scale(p.bits, p.constellation)
    for i in range(ids.size):
        res = O.frame_chain_masked(p, vt, vr, chans[:, ci[i]], snr[si[i]], sym[i].T, nz[i], roll_off=10)
        a, b = R.per_bin_errors(p, res, sym[i].T)
        want_s[si[i], ci[i]] += a
        want_b[si[i], ci[i]] += b
        x = res.eq / sc
        near = np.minimum(dist(x.real, m), dist(x.imag, m)) <= 1e-3 * np.maximum(1.0, np.abs(x))
        slack[si[i], ci[i]] += near.sum(axis=1)
    cells = np.zeros((2, Cn), dtype=np.int64)
    np.add.at(cells, (si, ci), 1)
    check_cells_and_totals(p, r, cells, True)
    assert want_s.sum() > 0
    assert np.all(np.abs(r["sym_err"] - want_s) <= slack), (np.abs(r["sym_err"] - want_s).max(), slack.max())
    assert np.all(np.abs(r["bit_err"] - want_b) <= 2 * slack), (np.abs(r["bit_err"] - want_b).max(), slack.max())


def mask_job():
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    vt, vr, _, _ = O.perturbed_windows(p, seed=4)
    return p, to_sys(p), vt, vr, O.synth_channels(4, 21, seed=5), np.array([0.0, 6.0, 12.0, 18.0])


@pytest.mark.gpu
@pytest.mark.parametrize("fft", [False, True])
def test_unreachable_target_is_the_fixed_run(handle, fft, clean_env):
    """Row 0 is ber_run_masked(ensemble_max, variant + 1) and row 1 ber_run(ensemble_max, variant), bit for bit."""
    if fft:
        clean_env.setenv("WOFDM_MASK_FFT", "1")
    p, s, vt, vr, chans, snr = mask_job()
    E, seed, variant = 6, 7, 2
    masked = handle.ber_run_masked(s, vt, vr, chans, snr, E, seed=seed, variant=variant + 1)
    plain = handle.ber_run(s, vt, vr, chans, snr, E, seed=seed, variant=variant)
    for kw in (dict(target_symbol_errors=10 ** 15), dict(target_bit_errors=10 ** 15, first_block=E)):
        r = handle.ber_run_masked_adaptive(s, vt, vr, chans, snr, E, seed=seed, variant=variant, **kw)
        assert np.array_equal(r["ensemble_used"], np.full(len(snr), E))
        assert r["rounds"] == (1 if "first_block" in kw else 3)                       # blocks 1, 2, 3
        for row, ref in enumerate((masked, plain)):
            assert np.array_equal(r["bit_err"][row], ref["bit_err"]) and np.array_equal(r["sym_err"][row], ref["sym_err"]), row
            assert np.array_equal(r["bit_tot"], ref["bit_tot"]) and np.array_equal(r["sym_tot"], ref["sym_tot"])
    assert masked["sym_err"].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [A.SYM, A.BIT])
def test_schedule_matches_oracle(handle, kind, clean_env):
    """Per-(point, e) counts of both chains from one-index segments, fed to oracle/adaptive.py with the two chains as its
    rows: the adaptive call returns its ensemble_used, counters and rounds exactly, with targets that stop the points in
    different rounds."""
    p, s, vt, vr, chans, snr = mask_job()
    E, seed = 16, 9
    bit = np.zeros((2, 4, E), dtype=np.int64)
    sym = np.zeros((2, 4, E), dtype=np.int64)
    for e in range(E):
        one_idx = [(k, e, 1) for k in range(4)]
        rm = handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, one_idx, seed=seed, variant=1)
        ru = handle.ber_run_segments(s, [vt], [vr], chans, snr, E, one_idx, seed=seed, variant=0)
        bit[0, :, e], sym[0, :, e] = rm["bit_err"], rm["sym_err"]
        bit[1, :, e], sym[1, :, e] = ru["bit_err"][0], ru["sym_err"][0]
    tab = bit if kind == A.BIT else sym
    m_all = tab.sum(axis=2).min(axis=0)
    assert m_all.min() > 0
    tested = set()
    for target in sorted({int(x) for x in np.geomspace(max(1, m_all.min() // 8), m_all.max(), 7)}):
        used, tb, ts, rounds, blocks = A.schedule(bit, sym, target, kind, first_block=1)
        stop_round = [max(i for i, rnd in enumerate(blocks) if k in rnd) for k in range(4)]
        r = handle.ber_run_masked_adaptive(s, vt, vr, chans, snr, E, first_block=1, seed=seed,
                                           **({"target_bit_errors": target} if kind == A.BIT else {"target_symbol_errors": target}))
        assert r["ensemble_used"].tolist() == used, (target, r["ensemble_used"], used)
        assert r["bit_err"].tolist() == tb and r["sym_err"].tolist() == ts and r["rounds"] == rounds, target
        assert np.array_equal(r["sym_tot"], np.asarray(used) * chans.shape[1] * int(p.active.sum()) * (p.S - 1))
        tested.add(len(set(stop_round)))
    assert max(tested) >= 3, "the targets must stop points in different rounds"


@pytest.mark.gpu
def test_shards_in_two_threads(clean_env):
    """Two handles on device 0, shards (0, 2) and (1, 2), summed by a threading.Barrier reducer: each returns the
    single-process result."""
    p, s, vt, vr, chans, snr = mask_job()
    with W.Handle([0]) as h0:
        first = h0.ber_run_masked_segments(s, vt, vr, chans, snr, 40, [(k, 0, 1) for k in range(len(snr))], seed=3, variant=1)
        kw = dict(target_symbol_errors=4 * int(first["sym_err"].max()) + 1, first_block=1, seed=3)
        want = h0.ber_run_masked_adaptive(s, vt, vr, chans, snr, 40, **kw)
    bar = threading.Barrier(2, timeout=300)
    slots, out = [None, None], [None, None]

    def reducer(rank):
        def red(counts):
            assert counts.shape == (2, len(snr), 2)
            slots[rank] = counts.copy()
            bar.wait()
            tot = slots[0] + slots[1]
            bar.wait()
            return tot
        return red

    def run(rank):
        with W.Handle([0]) as h:
            out[rank] = h.ber_run_masked_adaptive(s, vt, vr, chans, snr, 40, shard=(rank, 2), reduce=reducer(rank), **kw)
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


@pytest.mark.gpu
def test_errors_and_handle_survives(handle, clean_env):
    p, s, vt, vr, chans, snr = mask_job()
    E, EINVAL = 8, W.capi.EINVAL
    ref = handle.ber_run_masked(s, vt, vr, chans, snr, E, seed=2, variant=1)

    def still_works():
        r = handle.ber_run_masked_segments(s, vt, vr, chans, snr, E, [(k, 0, E) for k in range(4)], seed=2, variant=1)
        for key in ref:
            assert np.array_equal(r[key], ref[key]), key

    def seg_rc(segs, **kw):
        with pytest.raises(W.WofdmError) as ei:
            handle.ber_run_masked_segments(kw.pop("sys", s), vt, vr, chans, snr, kw.pop("E", E), segs, **kw)
        return ei.value.code
    assert seg_rc(np.zeros((0, 3))) == EINVAL                                   # n_seg < 1
    assert seg_rc([(4, 0, 1)]) == EINVAL and seg_rc([(-1, 0, 1)]) == EINVAL     # SNR index outside [0, n_snr)
    assert seg_rc([(0, 8, 1)]) == EINVAL and seg_rc([(0, -1, 2)]) == EINVAL     # e_begin outside [0, ensemble_max)
    assert seg_rc([(0, 6, 3)]) == EINVAL                                        # runs past ensemble_max
    assert seg_rc([(0, 2, 0)]) == EINVAL                                        # e_count < 1
    assert seg_rc([(1, 0, 4), (0, 0, 8), (1, 3, 2)]) == EINVAL                  # overlap within point 1
    assert seg_rc([(0, 0, 1)], E=0) == EINVAL                                   # ensemble_max < 1
    assert seg_rc([(0, 0, 1)], E=2 ** 62) == EINVAL                             # n_snr * C * ensemble_max overflows
    for bad in ((-1, 2), (2, 2), (0, 0), (3, 1)):
        assert seg_rc([(0, 0, 1)], shard=bad) == EINVAL
    assert seg_rc([(0, 0, 1)], sys=s.copy(precision=1)) == W.capi.EUNSUPPORTED  # fp64
    s64 = W.params_from_name("CP", 64, 8, 0, 0, bits=4, S=4, noise_norm=1, constellation=1)
    with pytest.raises(W.WofdmError) as ei:                                      # N outside {128, 256, 512}
        handle.ber_run_masked_segments(s64, np.ones(s64.n_tx), np.ones(64), chans, snr, E, [(0, 0, 1)])
    assert ei.value.code == W.capi.EUNSUPPORTED
    assert seg_rc([(0, 0, 1)], roll_off=0) == EINVAL
    still_works()
    # NULL segments / outputs, unknown resolve bits, an overflowing counter array through the C-ABI
    lib = W.capi.load()
    wta, wra = np.ascontiguousarray(vt), np.ascontiguousarray(vr)
    chf = np.ascontiguousarray(chans.T, dtype=np.complex128)
    snr_ = np.ascontiguousarray(snr)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    o = [np.zeros(4 * 4 * 256, dtype=np.int64) for _ in range(6)]
    segs = np.array([[0, 0, 1]], dtype=np.int64)

    def raw_seg(segp, n, res, outs=None, n_snr=4, n_chan=4):
        outs = outs if outs is not None else [ip(o[0]), ip(o[1]), ip(o[2])]
        return lib.wofdm_ber_run_masked_segments(handle._h, C.byref(s), dp(wta), dp(wra), dp(chf.view(np.float64)), 21, n_chan,
                                                 dp(snr_), n_snr, E, segp, n, 0, 1, 10, 0, 1, res, *outs)
    assert raw_seg(None, 1, 0) == EINVAL
    for res in (4, 5, -1):
        assert raw_seg(ip(segs), 1, res) == EINVAL
    for k in range(3):
        outs = [ip(o[0]), ip(o[1]), ip(o[2])]
        outs[k] = None
        assert raw_seg(ip(segs), 1, 0, outs) == EINVAL
    # 2^30 points x 2^30 channels x 256 bins x 16 bytes of counters overflow size_t (the check reads no input array)
    assert raw_seg(ip(segs), 1, 3, n_snr=1 << 30, n_chan=1 << 30) == EINVAL
    assert raw_seg(ip(segs), 1, 3) == W.capi.OK
    still_works()

    def ad_rc(**kw):
        with pytest.raises(W.WofdmError) as ei:
            handle.ber_run_masked_adaptive(kw.pop("sys", s), vt, vr, chans, snr, kw.pop("E", E), **kw)
        return ei.value.code
    assert ad_rc(target_symbol_errors=0) == EINVAL
    assert ad_rc(target_bit_errors=-5) == EINVAL
    assert ad_rc(target_symbol_errors=10, first_block=0) == EINVAL
    assert ad_rc(target_symbol_errors=10, E=0) == EINVAL
    assert ad_rc(target_symbol_errors=10, E=2 ** 62) == EINVAL
    assert ad_rc(target_symbol_errors=10, shard=(0, 2)) == EINVAL              # shard_count > 1 without reduce
    assert ad_rc(target_symbol_errors=10, shard=(2, 2), reduce=lambda c: None) == EINVAL
    assert ad_rc(target_symbol_errors=10, roll_off=0) == EINVAL
    assert ad_rc(target_symbol_errors=10, sys=s.copy(precision=1)) == W.capi.EUNSUPPORTED

    def boom(counts):
        raise RuntimeError("reduce failed")
    with pytest.raises(W.WofdmError) as ei:
        handle.ber_run_masked_adaptive(s, vt, vr, chans, snr, E, target_symbol_errors=10, reduce=boom)
    assert ei.value.code == EINVAL and isinstance(ei.value.__cause__, RuntimeError)
    with pytest.raises(W.WofdmError):                                            # neither / both targets
        handle.ber_run_masked_adaptive(s, vt, vr, chans, snr, E)
    used, rounds = np.zeros(4, dtype=np.int64), C.c_int(0)
    nul = W.capi.REDUCE_FN()

    def raw_ad(kind, outs=None):
        outs = outs if outs is not None else [ip(used), ip(o[0]), ip(o[1]), ip(o[2]), ip(o[3]), C.byref(rounds)]
        return lib.wofdm_ber_run_masked_adaptive(handle._h, C.byref(s), dp(wta), dp(wra), dp(chf.view(np.float64)), 21, 4,
                                                 dp(snr_), 4, E, 1, kind, 10, 0, 0, 10, 0, 1, nul, None, *outs)
    assert raw_ad(2) == EINVAL and raw_ad(-1) == EINVAL
    for k in range(6):
        outs = [ip(used), ip(o[0]), ip(o[1]), ip(o[2]), ip(o[3]), C.byref(rounds)]
        outs[k] = None
        assert raw_ad(W.capi.WOFDM_TARGET_SYMBOL_ERRORS, outs) == EINVAL
    assert raw_ad(W.capi.WOFDM_TARGET_SYMBOL_ERRORS) == W.capi.OK
    still_works()
    a = handle.ber_run_masked_adaptive(s, vt, vr, chans, snr, E, target_symbol_errors=50, seed=2)
    b = handle.ber_run_masked_adaptive(s, vt, vr, chans, snr, E, target_symbol_errors=50, seed=2, reduce=lambda c: None)
    for key in ("bit_err", "sym_err", "ensemble_used", "rounds"):
        assert np.array_equal(a[key], b[key]), key


@pytest.mark.gpu
def test_run_sim_mc_adaptive_mirror(handle, clean_env):
    """An unreachable target gives run_sim_mc's (berMasked, ber) at ensemble = ensemble_max for every channel row and SNR;
    a reachable one stops early."""
    from wofdm_b200 import ofdm_utils as U
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    vt, vr, _, _ = O.perturbed_windows(p, seed=16)
    ch = O.synth_channels(1, 21, seed=16)[:, 0]
    rest = (p.cp, p.cs, 8, 0, np.diag(vt), np.diag(vr), ch, 12.0, 64, p.rm, p.shift, 256, 4, 16, 10)
    bm, b0 = U.run_sim_mc(20, *rest, seed=3, handle=handle)
    am, a0, used = U.run_sim_mc_adaptive(20, *rest, target_bit_errors=10 ** 15, first_block=4, seed=3, handle=handle)
    assert am.shape == a0.shape == used.shape == (1,)
    assert am[0] == bm and a0[0] == b0 and used[0] == 20 and bm > 0
    chans = O.synth_channels(3, 21, seed=2).T                              # C x L, rows = realisations
    snrs = np.array([4.0, 12.0, 20.0])
    rest2 = rest[:6] + (chans, snrs) + rest[8:]
    am, a0, used = U.run_sim_mc_adaptive(30, *rest2, target_bit_errors=2000, seed=5, handle=handle)
    assert am.shape == a0.shape == used.shape == (3,) and used.min() < 30
    r = handle.ber_run_masked_adaptive(to_sys(p), vt, vr, chans.T, snrs, 30, target_bit_errors=2000, seed=5)
    assert np.array_equal(am, r["bit_err"][0] / r["bit_tot"]) and np.array_equal(a0, r["bit_err"][1] / r["bit_tot"])
