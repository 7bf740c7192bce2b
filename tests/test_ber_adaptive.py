"""Frame segments and the stopping rule of the BER chain (wofdm_ber_run_segments, wofdm_ber_run_adaptive).

CPU: the schedule of oracle/adaptive.py on synthetic count tables; the sharding.adaptive_allreduce trampoline called through
ctypes in a two-rank gloo group.
GPU (the policy table of test_ber_resolved.CASES): an unreachable target reproduces wofdm_ber_run_multi(ensemble_max);
segments add up to multi / resolved runs; the schedule equals the oracle's on measured per-index counts; an fp64 run is
replayed through the CPU oracle; shards in two threads and two devices give the single-process result; error codes; the
wOFDMSystem mirror.
"""
import ctypes as C
import os
import socket
import threading

import numpy as np
import pytest

import wofdm_b200 as W
from wofdm_b200 import sharding
from oracle import adaptive as A
from oracle import wofdm_oracle as O
from test_ber_resolved import CASES, kernel_of, to_sys, windows


# ---------------------------------------------------------------- CPU: the schedule

def cumulative_rounds(blocks):
    """per point: the cumulative ensemble indices after each of its rounds"""
    out = {}
    for rnd in blocks:
        for s, b in rnd.items():
            prev = out[s][-1] if s in out else 0
            out.setdefault(s, []).append(prev + b)
    return out


def test_schedule_stops_at_first_round_reaching_target():
    rng = np.random.default_rng(1)
    E, nv, ns = 64, 2, 5
    sym = rng.integers(0, 4, size=(nv, ns, E))
    sym[1] //= 2                                            # pair 1 is the slower one: it decides
    target = 20
    used, tb, ts, rounds, blocks = A.schedule(sym * 3, sym, target, A.SYM, first_block=1)
    cum = cumulative_rounds(blocks)
    for s in range(ns):
        m_at = [min(int(sym[v, s, :e].sum()) for v in range(nv)) for e in cum[s]]
        assert cum[s][-1] == used[s]
        assert all(m < target for m in m_at[:-1])           # not done earlier
        assert m_at[-1] >= target or used[s] == E           # done now
        for v in range(nv):
            assert ts[v][s] == int(sym[v, s, :used[s]].sum()) and tb[v][s] == 3 * ts[v][s]
    assert rounds == len(blocks)


def test_schedule_zero_errors_runs_to_ensemble_max_doubling():
    E = 100
    z = np.zeros((1, 2, E), dtype=np.int64)
    used, _, _, rounds, blocks = A.schedule(z, z, 5, A.BIT, first_block=3)
    assert used == [E, E]
    assert [r[0] for r in blocks] == [3, 6, 12, 24, 48, 7]   # doubling, the last block clipped at ensemble_max
    assert rounds == 6


def test_schedule_blocks_never_more_than_double():
    rng = np.random.default_rng(7)
    for trial in range(20):
        E = int(rng.integers(1, 300))
        cnt = rng.integers(0, 3, size=(2, 6, E)) * (rng.random((2, 6, 1)) < 0.8)
        used, _, _, _, blocks = A.schedule(cnt, cnt, int(rng.integers(1, 200)), A.SYM, first_block=int(rng.integers(1, 9)))
        prev = {}
        for rnd in blocks:
            for s, b in rnd.items():
                assert 1 <= b and (s not in prev or b <= 2 * prev[s])
                prev[s] = b
        assert all(1 <= u <= E for u in used)


def test_schedule_first_block_covers_ensemble_max():
    cnt = np.ones((2, 3, 10), dtype=np.int64)
    for fb in (10, 11, 10 ** 6):
        used, _, _, rounds, _ = A.schedule(cnt, cnt, 10 ** 9, A.SYM, first_block=fb)
        assert rounds == 1 and used == [10, 10, 10]


def test_schedule_128_bit_products():
    """target * e beyond 2^64: the next block is the exact ceil((target - m) * e / m), clipped by 2b and ensemble_max."""
    class Const:                                            # a huge ensemble without materialising its counts
        def __init__(self, v, n):
            self.v, self.n = v, n

        def __len__(self):
            return self.n

        def range_sum(self, lo, hi):
            return self.v * (min(hi, self.n) - lo)
    E = 2 ** 62
    target = 2 ** 61
    cnt = [[Const(1, E)]]
    used, _, ts, rounds, blocks = A.schedule(cnt, cnt, target, A.SYM, first_block=2 ** 40, ensemble_max=E)
    # round 0: 2^40 indices, m = 2^40 errors; need = ceil((2^61 - 2^40) * 2^40 / 2^40) = 2^61 - 2^40 > 2b = 2^41
    assert blocks[1][0] == 2 ** 41
    assert (target - 2 ** 40) * 2 ** 40 > 2 ** 64             # the product the library must form in 128 bits
    assert used[0] >= target and ts[0][0] == used[0] and used[0] <= E
    # the last block is the exact remainder once doubling would overshoot
    cum = cumulative_rounds(blocks)[0]
    assert cum[-1] == target and cum[-2] < target


# ---------------------------------------------------------------- CPU: the reduce trampoline under gloo

def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cb = W.capi.reduce_trampoline(sharding.adaptive_allreduce(), (2, 3, 2))
    counts = (np.arange(12, dtype=np.int64) + 1) * (rank + 1)
    rc = cb(counts.ctypes.data_as(C.POINTER(C.c_int64)), counts.size, None)     # through the C function pointer
    bad = W.capi.reduce_trampoline(lambda a: np.zeros(5))
    rc_bad = bad(counts.ctypes.data_as(C.POINTER(C.c_int64)), counts.size, None)
    q.put((rank, rc, counts.copy(), rc_bad, cb.error))
    dist.barrier()
    dist.destroy_process_group()


def test_adaptive_allreduce_trampoline_two_ranks():
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = (np.arange(12, dtype=np.int64) + 1) * 3
    for _, rc, counts, rc_bad, err in got:
        assert rc == 0 and err is None
        assert np.array_equal(counts, want)
        assert rc_bad != 0                                  # a wrong-sized result fails the call instead of passing silently


def test_segment_frame_ids_launch_order():
    segs = [(1, 2, 2), (0, 0, 1)]
    f = sharding.segment_frame_ids(segs, 3, 5)
    assert f.tolist() == [17, 18, 22, 23, 27, 28, 0, 5, 10]
    assert sharding.segment_frame_ids(segs, 3, 5, shard=(1, 2)).tolist() == [18, 23, 28, 5]
    si, c, e = sharding.decode(f, 3, 5)
    assert si.tolist() == [1] * 6 + [0] * 3 and e.tolist() == [2, 3, 2, 3, 2, 3, 0, 0, 0]


# ---------------------------------------------------------------- GPU

@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def setup_case(case, monkeypatch):
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
    return p, s, [w[0] for w in wins], [w[1] for w in wins], chans, snr, kern, wins


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_unreachable_target_is_the_fixed_run(handle, case, monkeypatch):
    p, s, wt, wr, chans, snr, kern, wins = setup_case(case, monkeypatch)
    assert kern in kernel_of(handle, s, wins, chans, snr)
    E = 6
    ref = handle.ber_run_multi(s, wt, wr, chans, snr, E, seed=p.N + 1, variant=3)
    for kw in (dict(target_symbol_errors=10 ** 15), dict(target_bit_errors=10 ** 15)):
        r = handle.ber_run_adaptive(s, wt, wr, chans, snr, E, first_block=1, seed=p.N + 1, variant=3, **kw)
        assert np.array_equal(r["ensemble_used"], np.full(len(snr), E)) and r["rounds"] == 3     # blocks 1, 2, 3
        assert np.array_equal(r["sym_tot"], ref["sym_tot"]) and np.array_equal(r["bit_tot"], ref["bit_tot"])
        assert np.array_equal(r["sym_err"], ref["sym_err"]) and np.array_equal(r["bit_err"], ref["bit_err"]), case
    assert ref["sym_err"].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_segments_add_up(handle, case, monkeypatch):
    """[0, e1) and [e1, E) out of order and interleaved across points: in one call, and split over two calls, they give
    multi(E) unresolved and ber_run_resolved(E) for every resolution."""
    p, s, wt, wr, chans, snr, kern, wins = setup_case(case, monkeypatch)
    E, e1, seed = 7, 3, 11
    lo = [(k, 0, e1) for k in range(3)]
    hi = [(k, e1, E - e1) for k in range(3)]
    one_call = [hi[2], lo[0], hi[1], lo[2], hi[0], lo[1]]
    split = ([hi[1], lo[0], lo[2]], [lo[1], hi[2], hi[0]])
    ref = handle.ber_run_multi(s, wt, wr, chans, snr, E, seed=seed, variant=1)
    seg = lambda sg, **kw: handle.ber_run_segments(s, wt, wr, chans, snr, E, sg, seed=seed, variant=1, **kw)
    r = seg(one_call)
    parts = [seg(x) for x in split]
    for key in ("bit_err", "sym_err"):
        assert np.array_equal(r[key], ref[key]), (case, key)
        assert np.array_equal(parts[0][key] + parts[1][key], ref[key]), (case, key)
    assert np.array_equal(r["sym_tot"], ref["sym_tot"]) and np.array_equal(parts[0]["sym_tot"] + parts[1]["sym_tot"], ref["sym_tot"])
    for bins, chan in ((True, False), (False, True), (True, True)):
        rr = handle.ber_run_resolved(s, wt, wr, chans, snr, E, seed=seed, variant=1, by_subcarrier=bins, by_channel=chan)
        a = seg(split[0], by_subcarrier=bins, by_channel=chan)
        b = seg(split[1], by_subcarrier=bins, by_channel=chan)
        for key in ("bit_err", "sym_err", "sym_tot"):
            assert a[key].shape == rr[key].shape
            assert np.array_equal(a[key] + b[key], rr[key]), (case, bins, chan, key)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [A.SYM, A.BIT])
def test_schedule_matches_oracle(handle, kind, monkeypatch):
    """Per-(point, e) counts from 16 one-index segment calls, fed to oracle/adaptive.py: the adaptive call must return its
    ensemble_used, counters and rounds exactly, with targets that stop the points in different rounds."""
    monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    p = O.system_params("WOLA", 256, 16, 8, 10, S=16, bits=4)
    s = to_sys(p, 0)
    wins = windows(p, 2, seed=4)
    wt, wr = [w[0] for w in wins], [w[1] for w in wins]
    chans = O.synth_channels(4, 21, seed=5)
    snr = np.array([0.0, 6.0, 12.0, 18.0])
    E, seed = 16, 9
    bit = np.zeros((2, 4, E), dtype=np.int64)
    sym = np.zeros((2, 4, E), dtype=np.int64)
    for e in range(E):
        r = handle.ber_run_segments(s, wt, wr, chans, snr, E, [(k, e, 1) for k in range(4)], seed=seed)
        bit[:, :, e], sym[:, :, e] = r["bit_err"], r["sym_err"]
    tab = bit if kind == A.BIT else sym
    m_all = tab.sum(axis=2).min(axis=0)                     # the fewest errors of each point over the whole ensemble
    assert m_all.min() > 0
    tested = set()
    for target in sorted({int(x) for x in np.geomspace(max(1, m_all.min() // 8), m_all.max(), 7)}):
        used, tb, ts, rounds, blocks = A.schedule(bit, sym, target, kind, first_block=1)
        stop_round = [max(i for i, rnd in enumerate(blocks) if k in rnd) for k in range(4)]
        r = handle.ber_run_adaptive(s, wt, wr, chans, snr, E, first_block=1, seed=seed,
                                    **({"target_bit_errors": target} if kind == A.BIT else {"target_symbol_errors": target}))
        assert r["ensemble_used"].tolist() == used, (target, r["ensemble_used"], used)
        assert r["bit_err"].tolist() == tb and r["sym_err"].tolist() == ts and r["rounds"] == rounds, target
        assert np.array_equal(r["sym_tot"], np.asarray(used) * chans.shape[1] * p.N * (p.S - 1))
        tested.add(len(set(stop_round)))
    assert max(tested) >= 3, "the targets must stop points in different rounds"


@pytest.mark.gpu
def test_fp64_run_replays_through_cpu_oracle(handle):
    """The frames an fp64 adaptive run used (segment_frame_ids of {s, 0, ensemble_used[s]}), exported with wofdm_ber_draws
    and decided by the CPU oracle: the per-frame counts sum to the run's counters exactly."""
    p = O.system_params("WOLA", 64, 8, 4, 4, S=8, bits=4)
    s = to_sys(p, 1)
    wins = windows(p, 2, seed=8)
    wt, wr = [w[0] for w in wins], [w[1] for w in wins]
    L, Cn, E, seed, variant = 5, 2, 6, 13, 4
    chans = O.synth_channels(Cn, L, seed=3)
    snr = np.array([2.0, 12.0, 30.0])
    r = handle.ber_run_adaptive(s, wt, wr, chans, snr, E, target_symbol_errors=40, seed=seed, variant=variant)
    used = r["ensemble_used"]
    assert used.min() < E and used.max() == E and r["sym_err"].sum() > 0        # points stopped early and at ensemble_max
    ids = sharding.segment_frame_ids([(k, 0, int(u)) for k, u in enumerate(used)], Cn, E)
    si, ci, _ = sharding.decode(ids, Cn, E)
    want_b = np.zeros((2, len(snr)), dtype=np.int64)
    want_s = np.zeros((2, len(snr)), dtype=np.int64)
    for v in range(2):
        sym, nz = handle.ber_draws(s, L, seed, variant + v, ids)
        for i in range(ids.size):
            res = O.frame_chain_structured(p, wt[v], wr[v], chans[:, ci[i]], snr[si[i]], sym[i].T, nz[i])
            want_b[v, si[i]] += res.bit_err
            want_s[v, si[i]] += res.sym_err
    assert np.array_equal(r["sym_err"], want_s) and np.array_equal(r["bit_err"], want_b)


def small_job(p_name="WOLA"):
    p = O.system_params(p_name, 256, 16, 8, 10, S=16, bits=4)
    s = to_sys(p, 0)
    wins = windows(p, 2, seed=6)
    return p, s, [w[0] for w in wins], [w[1] for w in wins], O.synth_channels(5, 21, seed=7), np.array([0.0, 8.0, 16.0])


@pytest.mark.gpu
def test_shards_in_two_threads(monkeypatch):
    """Two handles on device 0, shards (0, 2) and (1, 2), summed by a threading.Barrier reducer: each returns the
    single-process result (ctypes releases the GIL during the call)."""
    monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    p, s, wt, wr, chans, snr = small_job()
    with W.Handle([0]) as h0:
        # a target no point reaches with its first ensemble index, so that the schedule takes several rounds
        first = h0.ber_run_segments(s, wt, wr, chans, snr, 40, [(k, 0, 1) for k in range(len(snr))], seed=3)
        m0 = first["sym_err"].min(axis=0)
        assert m0.max() > 0
        kw = dict(target_symbol_errors=4 * int(m0.max()) + 1, first_block=1, seed=3)
        want = h0.ber_run_adaptive(s, wt, wr, chans, snr, 40, **kw)
    bar = threading.Barrier(2, timeout=300)
    slots, out = [None, None], [None, None]

    def reducer(rank):
        def red(counts):
            slots[rank] = counts.copy()
            bar.wait()
            tot = slots[0] + slots[1]
            bar.wait()
            return tot
        return red

    def run(rank):
        with W.Handle([0]) as h:
            out[rank] = h.ber_run_adaptive(s, wt, wr, chans, snr, 40, shard=(rank, 2), reduce=reducer(rank), **kw)
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
def test_two_device_handle_matches_one_device(handle):
    n = C.c_int(0)
    assert W.capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("one visible device")
    p, s, wt, wr, chans, snr = small_job()
    kw = dict(target_bit_errors=2000, seed=5)
    one = handle.ber_run_adaptive(s, wt, wr, chans, snr, 30, **kw)
    with W.Handle([0, 1]) as h2:
        two = h2.ber_run_adaptive(s, wt, wr, chans, snr, 30, **kw)
        seg2 = h2.ber_run_segments(s, wt, wr, chans, snr, 30, [(1, 3, 5), (0, 0, 2)], seed=5, by_channel=True)
    seg1 = handle.ber_run_segments(s, wt, wr, chans, snr, 30, [(1, 3, 5), (0, 0, 2)], seed=5, by_channel=True)
    for key in ("bit_err", "sym_err", "sym_tot", "ensemble_used", "rounds"):
        assert np.array_equal(one[key], two[key]), key
    for key in ("bit_err", "sym_err", "sym_tot"):
        assert np.array_equal(seg1[key], seg2[key]), key


@pytest.mark.gpu
def test_errors_and_handle_survives(handle):
    p, s, wt, wr, chans, snr = small_job()
    E = 8
    EINVAL = W.capi.EINVAL

    def seg_rc(segs, **kw):
        with pytest.raises(W.WofdmError) as ei:
            handle.ber_run_segments(s, wt, wr, chans, snr, kw.pop("E", E), segs, **kw)
        return ei.value.code
    assert seg_rc(np.zeros((0, 3))) == EINVAL                                   # n_seg < 1
    assert seg_rc([(3, 0, 1)]) == EINVAL and seg_rc([(-1, 0, 1)]) == EINVAL     # SNR index outside [0, n_snr)
    assert seg_rc([(0, 8, 1)]) == EINVAL and seg_rc([(0, -1, 2)]) == EINVAL     # e_begin outside [0, ensemble_max)
    assert seg_rc([(0, 6, 3)]) == EINVAL                                        # runs past ensemble_max
    assert seg_rc([(0, 2, 0)]) == EINVAL                                        # e_count < 1
    assert seg_rc([(1, 0, 4), (0, 0, 8), (1, 3, 2)]) == EINVAL                  # overlap within point 1
    assert seg_rc([(0, 0, 1)], E=0) == EINVAL                                   # ensemble_max < 1
    assert seg_rc([(0, 0, 1)], E=2 ** 62) == EINVAL                             # n_snr * C * ensemble_max overflows
    assert seg_rc([(0, 0, 1)], by_subcarrier=True, shard=(2, 2)) == EINVAL       # what _resolved rejects
    # NULL segments / an unknown resolve bit through the C-ABI
    lib = W.capi.load()
    wta, wra = np.ascontiguousarray(wt), np.ascontiguousarray(wr)
    chf = np.ascontiguousarray(chans.T, dtype=np.complex128)
    snr_ = np.ascontiguousarray(snr)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    o = [np.zeros(2 * 3 * 256 * 5, dtype=np.int64) for _ in range(6)]
    segs = np.array([[0, 0, 1]], dtype=np.int64)
    raw_seg = lambda segp, n, res: lib.wofdm_ber_run_segments(handle._h, C.byref(s), dp(wta), dp(wra), 2, dp(chf.view(np.float64)), 21, 5,
                                                              dp(snr_), 3, E, segp, n, 0, 0, 0, 1, res, ip(o[0]), ip(o[1]), ip(o[2]))
    assert raw_seg(None, 1, 0) == EINVAL and raw_seg(ip(segs), 1, 4) == EINVAL
    assert raw_seg(ip(segs), 1, 3) == W.capi.OK

    def ad_rc(**kw):
        with pytest.raises(W.WofdmError) as ei:
            handle.ber_run_adaptive(s, wt, wr, chans, snr, kw.pop("E", E), **kw)
        return ei.value.code
    assert ad_rc(target_symbol_errors=0) == EINVAL
    assert ad_rc(target_bit_errors=-5) == EINVAL
    assert ad_rc(target_symbol_errors=10, first_block=0) == EINVAL
    assert ad_rc(target_symbol_errors=10, E=0) == EINVAL
    assert ad_rc(target_symbol_errors=10, E=2 ** 62) == EINVAL
    assert ad_rc(target_symbol_errors=10, shard=(0, 2)) == EINVAL              # shard_count > 1 without reduce

    def boom(counts):
        raise RuntimeError("reduce failed")
    with pytest.raises(W.WofdmError) as ei:
        handle.ber_run_adaptive(s, wt, wr, chans, snr, E, target_symbol_errors=10, reduce=boom)
    assert ei.value.code == EINVAL and isinstance(ei.value.__cause__, RuntimeError)
    with pytest.raises(W.WofdmError):                                            # neither / both targets
        handle.ber_run_adaptive(s, wt, wr, chans, snr, E)
    used, rounds = np.zeros(3, dtype=np.int64), C.c_int(0)
    nul = W.capi.REDUCE_FN()
    raw_ad = lambda kind: lib.wofdm_ber_run_adaptive(handle._h, C.byref(s), dp(wta), dp(wra), 2, dp(chf.view(np.float64)), 21, 5,
                                                     dp(snr_), 3, E, 1, kind, 10, 0, 0, 0, 1, nul, None, ip(used), ip(o[0]),
                                                     ip(o[1]), ip(o[2]), ip(o[3]), C.byref(rounds))
    assert raw_ad(2) == EINVAL and raw_ad(-1) == EINVAL
    assert raw_ad(W.capi.WOFDM_TARGET_SYMBOL_ERRORS) == W.capi.OK
    # the handle still works, and an identity reduce changes nothing
    a = handle.ber_run_adaptive(s, wt, wr, chans, snr, E, target_symbol_errors=50, seed=2)
    b = handle.ber_run_adaptive(s, wt, wr, chans, snr, E, target_symbol_errors=50, seed=2, reduce=lambda c: None)
    for key in ("bit_err", "sym_err", "ensemble_used", "rounds"):
        assert np.array_equal(a[key], b[key]), key


@pytest.mark.gpu
def test_wofdm_system_mirror(handle):
    from wofdm_b200 import ofdm_utils as U
    chans = O.synth_channels(4, 21, seed=4)
    snr = np.array([0.0, 8.0, 16.0])
    for name, cp, ttx, trx in (("WOLA", 16, 8, 10), ("CP", 16, 0, 0)):
        sysm = U.wOFDMSystem(name, 256, cp, ttx, trx, "/nonexistent-folder", seed=11, handle=handle)
        p = O.system_params(name, 256, cp, ttx, trx, S=16)
        vt, vr, _, _ = O.perturbed_windows(p, seed=2)
        got = sysm.run_simulation_adaptive(chans, np.diag(vt), np.diag(vr), 20, snr, 16, 200, first_block=2)
        s = sysm._sys(16)
        if name == "CP":
            wt, wr = [np.ones(s.n_tx)], [np.ones(s.N + s.tail_rx)]
        else:
            wt, wr = [vt, W.capi.rc_window_tx(s)], [vr, W.capi.rc_window_rx(s)]
        r = handle.ber_run_adaptive(s, wt, wr, chans, snr, 20, target_symbol_errors=200, first_block=2, seed=11)
        want = [e / r["sym_tot"] for e in r["sym_err"]] + [r["ensemble_used"]]
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert np.array_equal(a, b)
        assert r["ensemble_used"].min() < 20
