"""Frame segments and resolved counters of the channel-mask chain for several window pairs and roll-offs in one call
(wofdm_ber_run_masked_segments_multi, Handle.ber_run_masked_segments_multi).

GPU: pair v's arrays equal ber_run_masked_segments with pair v's windows, roll-off and variant + v, bit for bit, for every
resolve on every path the masked chain takes (the shapes of test_ber_masked_multi.py, and the per-symbol FFT mask), across
product batches and shards; one whole-job segment per point is ber_run_masked_resolved per pair; disjoint segment lists
add up to ber_run_masked_multi; the refusals leave the handle usable; a two-device handle gives the one-device counters.
"""
import ctypes as C

import numpy as np
import pytest

import wofdm_b200 as W
from oracle import wofdm_oracle as O
from test_ber_masked_multi import CASES, ROLL_OFFS, clean_env, pairs, to_sys  # noqa: F401 -- clean_env is a fixture

SUB, CHAN = W.capi.WOFDM_BY_SUBCARRIER, W.capi.WOFDM_BY_CHANNEL
RESOLVES = {"none": (False, False), "sub": (True, False), "chan": (False, True), "sub_chan": (True, True)}


@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def check_against_singles(handle, s, wt, wr, ro, chans, snr, E, segs, seed=5, variant=3, shard=(0, 1), by_subcarrier=False,
                          by_channel=False):
    kw = dict(seed=seed, shard=shard, by_subcarrier=by_subcarrier, by_channel=by_channel)
    m = handle.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, segs, variant=variant, roll_offs=ro, **kw)
    n_var = len(ro)
    assert m["bit_err"].shape == m["sym_err"].shape == (n_var,) + m["sym_tot"].shape
    for v in range(n_var):
        r = handle.ber_run_masked_segments(s, wt[v], wr[v], chans, snr, E, segs, variant=variant + v, roll_off=ro[v], **kw)
        assert np.array_equal(m["bit_err"][v], r["bit_err"]), v
        assert np.array_equal(m["sym_err"][v], r["sym_err"]), v
        assert np.array_equal(m["sym_tot"], r["sym_tot"]) and np.array_equal(m["bit_tot"], r["bit_tot"])
    if n_var > 1:       # a mix-up of pairs cannot pass
        flat = m["bit_err"].reshape(n_var, -1)
        assert len({tuple(row) for row in flat}) == n_var, flat.sum(axis=1)
        assert np.all(flat.sum(axis=1) > 0)
    return m


SEGS = [(1, 3, 20), (0, 0, 15), (1, 30, 10), (0, 25, 15)]


@pytest.mark.gpu
@pytest.mark.parametrize("resolve", list(RESOLVES))
@pytest.mark.parametrize("case", list(CASES))
def test_pairs_equal_single_calls(handle, case, resolve, clean_env):
    name, N, cp, ttx, trx, bits, S, L, guard, n_var = CASES[case]
    p = O.system_params(name, N, cp, ttx, trx, S=S, bits=bits, noise_norm=1, constellation=1, guard=guard)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, n_var)
    sub, chan = RESOLVES[resolve]
    check_against_singles(handle, s, wt, wr, ro, O.synth_channels(3, L, seed=N + L), [6.0, 14.0], 40, SEGS,
                          by_subcarrier=sub, by_channel=chan)


@pytest.mark.gpu
@pytest.mark.parametrize("resolve", ["none", "sub_chan"])
def test_mask_fft_path(handle, resolve, clean_env):
    clean_env.setenv("WOFDM_MASK_FFT", "1")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 3)
    sub, chan = RESOLVES[resolve]
    check_against_singles(handle, s, wt, wr, ro, O.synth_channels(2, 21, seed=9), [6.0, 14.0], 40, SEGS,
                          by_subcarrier=sub, by_channel=chan)


@pytest.mark.gpu
def test_more_than_one_batch_and_shards(handle, clean_env):
    """17 000 local frames (more than the product's batch of 16 384) in 8 pairs, by sub-carrier; shards (k, 3) each against
    the single calls, and the three shards add up to the whole list."""
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 8)
    chans = O.synth_channels(5, 21, seed=6)
    snr, E = [4.0, 10.0], 2000
    segs = [(1, 300, 1700), (0, 0, 1700)]
    full = check_against_singles(handle, s, wt, wr, ro, chans, snr, E, segs, by_subcarrier=True)
    acc = {k: np.zeros_like(v) for k, v in full.items()}
    for k in range(3):
        part = check_against_singles(handle, s, wt, wr, ro, chans, snr, E, segs, shard=(k, 3), by_subcarrier=True)
        for key in acc:
            acc[key] += part[key]
    for key in acc:
        assert np.array_equal(acc[key], full[key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["gather_n256_v8", "staged_n128"])
def test_whole_job_segments_are_the_resolved_call(handle, case, clean_env):
    """One segment {s, 0, E} per point, by sub-carrier: pair v is ber_run_masked_resolved with its pair, bit for bit."""
    name, N, cp, ttx, trx, bits, S, L, guard, n_var = CASES[case]
    p = O.system_params(name, N, cp, ttx, trx, S=S, bits=bits, noise_norm=1, constellation=1, guard=guard)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, n_var)
    chans, snr, E = O.synth_channels(3, L, seed=4), [5.0, 12.0, 20.0], 30
    m = handle.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, [(k, 0, E) for k in range(3)], seed=8, variant=2,
                                             roll_offs=ro, by_subcarrier=True)
    for v in range(n_var):
        r = handle.ber_run_masked_resolved(s, wt[v], wr[v], chans, snr, E, seed=8, variant=2 + v, roll_off=ro[v],
                                           by_subcarrier=True)
        for key in ("bit_err", "sym_err"):
            assert np.array_equal(m[key][v], r[key]), (v, key)
        assert np.array_equal(m["sym_tot"], r["sym_tot"])


@pytest.mark.gpu
def test_disjoint_lists_add_up_to_the_multi_run(handle, clean_env):
    p = O.system_params("WOLA", 256, 22, 8, 10, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 4)
    chans, snr, E, e1 = O.synth_channels(4, 21, seed=3), [3.0, 9.0], 25, 11
    full = handle.ber_run_masked_multi(s, wt, wr, chans, snr, E, seed=6, variant=1, roll_offs=ro)
    a = handle.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, [(0, 0, e1), (1, 0, e1)], seed=6, variant=1, roll_offs=ro)
    b = handle.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, [(1, e1, E - e1), (0, e1, E - e1)], seed=6, variant=1,
                                             roll_offs=ro)
    for key in ("bit_err", "sym_err", "sym_tot", "bit_tot"):
        assert np.array_equal(a[key] + b[key], full[key]), key


def _raw(handle, s, wt, wr, chans, ro, n_var, segs, outs=True):
    wt, wr = np.ascontiguousarray(wt, dtype=np.float64), np.ascontiguousarray(wr, dtype=np.float64)
    chf = np.ascontiguousarray(np.asarray(chans, dtype=np.complex128).T)       # [C][L]
    L, Cn = chans.shape
    snr = np.array([6.0, 12.0])
    seg = np.ascontiguousarray(np.asarray(segs, dtype=np.int64).reshape(-1, 3))
    o = [np.zeros(max(1, 8 * 2), dtype=np.int64) for _ in range(3)]
    rop = None if ro is None else np.ascontiguousarray(ro, dtype=np.int32).ctypes.data_as(C.POINTER(C.c_int))
    return W.capi.load().wofdm_ber_run_masked_segments_multi(
        handle._h, C.byref(s), wt.ctypes.data_as(W.capi._dp), wr.ctypes.data_as(W.capi._dp), rop, n_var,
        chf.ctypes.data_as(W.capi._dp), L, Cn, snr.ctypes.data_as(W.capi._dp), 2, 10, seg.ctypes.data_as(W.capi._i64p),
        seg.shape[0], 1, 0, 0, 1, 0, *[(x.ctypes.data_as(W.capi._i64p) if outs else None) for x in o])


@pytest.mark.gpu
def test_refusals_leave_the_handle_usable(handle, clean_env):
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 8)
    wt9, wr9 = np.vstack([wt, wt[:1]]), np.vstack([wr, wr[:1]])
    chans = O.synth_channels(2, 21, seed=1)
    segs = [(0, 0, 5), (1, 2, 3)]
    EINVAL = W.capi.EINVAL
    want = handle.ber_run_masked_segments_multi(s, wt[:2], wr[:2], chans, [6.0, 12.0], 10, segs, seed=1, roll_offs=ro[:2])
    cases = [
        dict(n_var=0),
        dict(wt=wt9, wr=wr9, ro=ROLL_OFFS + [4], n_var=9),
        dict(ro=None),
        dict(ro=[4, 1000]),                                 # the second roll-off does not fit the mask
        dict(segs=[(0, 0, 5), (0, 4, 3)]),                  # overlapping segments of one point
        dict(outs=False),
    ]
    for kw in cases:
        args = dict(wt=wt[:2], wr=wr[:2], ro=ro[:2], n_var=2, segs=segs)
        args.update(kw)
        assert _raw(handle, s, args["wt"], args["wr"], chans, args["ro"], args["n_var"], args["segs"],
                    outs=args.get("outs", True)) == EINVAL, kw
        again = handle.ber_run_masked_segments_multi(s, wt[:2], wr[:2], chans, [6.0, 12.0], 10, segs, seed=1, roll_offs=ro[:2])
        for key in want:
            assert np.array_equal(again[key], want[key]), (kw, key)


@pytest.mark.gpu
def test_two_device_handle_matches_one_device(handle, clean_env):
    n = C.c_int(0)
    assert W.capi.load().wofdm_device_count(C.byref(n)) == 0
    if n.value < 2:
        pytest.skip("needs two GPUs")
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s = to_sys(p)
    wt, wr, ro = pairs(p, s, 3)
    chans, snr, E = O.synth_channels(4, 21, seed=2), [5.0, 11.0], 200
    segs = [(1, 0, 150), (0, 20, 180)]
    one = handle.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, segs, seed=4, roll_offs=ro, by_channel=True)
    with W.Handle([0, 1]) as h2:
        two = h2.ber_run_masked_segments_multi(s, wt, wr, chans, snr, E, segs, seed=4, roll_offs=ro, by_channel=True)
    for key in one:
        assert np.array_equal(one[key], two[key]), key
