"""A frame's error counts depend on (seed, global frame id, window pair) alone -- not on which CTA decides it, nor on how many
frames that CTA decided before.  Sharding, the multi-device handle, frame segments and the adaptive stopping rule all add
up disjoint frame sets on that promise (DESIGN section 6).

Every row of ROWS runs one reference job with wofdm_ber_run_multi and the same frames reassigned to other CTAs: the same call
again, one resident CTA per SM, shards summed (K = 2 and 47), a shuffled list of random segments over several calls, the
resolved counters and their shards, each window pair alone, a handle that owns every device.  Every counter must equal the
reference bit for bit; there is no tolerance in this file.  The fp32 tensor-core and register rows decide at least 3e8
symbols per reassignment at low SNR (SER 0.1 .. 0.7), where an arithmetic that depends on the assignment flips a decision
every ~1e7.  test_oracle_anchor replays frames that their CTA decided after many others through the CPU oracle, so that the
invariance is not that of a wrong answer.
"""
import ctypes
import re

import numpy as np
import pytest

import wofdm_b200 as W
from oracle import wofdm_oracle as O
from test_ber_gpu import flip_budget

pytestmark = pytest.mark.gpu

# name, N, cp, tail_tx, tail_rx, bits, L, pairs, precision, environment, kernel substrings ("!x": x absent), conv / noise_norm,
# guard, C, ensemble
ROWS = {
    "tconv2_n256": ("WOLA", 256, 16, 8, 10, 4, 21, 1, 0, {}, ["f32t2_n256"], 0, 0, 4, 10000),
    "tconv2_n256_3pairs": ("wtx", 256, 16, 8, 0, 4, 21, 3, 0, {}, ["f32t2_n256"], 1, 0, 4, 3500),
    "tconv2_n256_l84": ("WOLA", 256, 16, 8, 10, 4, 84, 2, 0, {}, ["f32t2_n256", "_l84"], 1, 0, 4, 5000),
    "tconv2_n512": ("CPW", 512, 32, 16, 20, 4, 21, 2, 0, {}, ["f32t2_n512"], 1, 0, 4, 2500),
    "tconv2_n1024": ("WOLA", 1024, 64, 32, 40, 6, 21, 2, 0, {}, ["f32t2_n1024", "_cl2"], 0, 0, 4, 10000),
    "tconv2_n1024_l84": ("CPW", 1024, 64, 32, 40, 6, 84, 1, 0, {}, ["f32t2_n1024", "_l84"], 1, 0, 4, 20000),
    "tconv1_n256": ("WOLA", 256, 16, 8, 10, 4, 21, 1, 0, {"WOFDM_TCONV_GEN": "1"}, ["ber_f32t_n256"], 0, 0, 4, 10000),
    "regs_n256_exact_fit": ("WOLA", 256, 16, 8, 10, 4, 21, 1, 0, {"WOFDM_NO_TCONV": "1"}, ["ber_f32r_n256", "_ftrue", "!_circ"], 1, 0, 4, 10000),
    "regs_n256_circ": ("wrx", 256, 16, 0, 10, 4, 21, 1, 0, {"WOFDM_NO_TCONV": "1"}, ["ber_f32r_n256", "_circ"], 0, 0, 4, 10000),
    "regs_n512": ("WOLA", 512, 32, 16, 20, 4, 21, 2, 0, {"WOFDM_NO_TCONV": "1"}, ["ber_f32r_n512"], 0, 0, 4, 2500),
    "regs_n1024_cluster": ("CPW", 1024, 64, 32, 40, 6, 21, 2, 0, {"WOFDM_NO_TCONV": "1"}, ["ber_f32r_n1024", "_cl2"], 1, 0, 4, 2500),
    "staged_n64": ("WOLA", 64, 8, 4, 4, 4, 5, 2, 0, {}, ["_c0_"], 0, 0, 4, 1250),
    "fp64_n256": ("WOLA", 256, 16, 8, 10, 4, 21, 2, 1, {}, ["f64_n256"], 1, 0, 4, 250),
    "fp64_n1024": ("WOLA", 1024, 64, 32, 40, 6, 21, 1, 1, {}, ["f64_n1024"], 0, 0, 4, 125),
    "guard_tconv2_n256": ("CPW", 256, 22, 8, 10, 4, 21, 2, 0, {}, ["f32t2_n256"], 1, 64, 4, 10000),
    "guard_tconv2_n1024": ("WOLA", 1024, 64, 32, 40, 6, 21, 1, 0, {}, ["f32t2_n1024"], 1, 256, 4, 20000),
}
BIG = 3e8                                    # decisions per reassignment of the fp32 tensor-core and register rows
ENV = ("WOFDM_NO_TCONV", "WOFDM_TCONV_GEN", "WOFDM_MAX_CTAS_PER_SM", "WOFDM_DEBUG")


@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def to_sys(p, precision):
    return W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift,
                  bits=p.bits, S=p.S, noise_norm=p.noise_norm, constellation=p.constellation, precision=precision,
                  guard=p.guard)


def low_snr(bits):
    """two points at a symbol error rate of ~0.15 .. 0.5 (most symbols near a decision boundary)"""
    return np.array([12.0, 18.0]) + (6.0 if bits == 6 else 0.0)


def set_env(monkeypatch, env):
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def plan_residency(handle, s, wt, wr, chans, snr, monkeypatch, capfd):
    """(kernel name, resident CTAs per SM, CTAs per frame) of the plan a job of these inputs runs (WOFDM_DEBUG report)."""
    monkeypatch.setenv("WOFDM_DEBUG", "1")
    capfd.readouterr()
    plan = handle.ber_plan_multi(s, wt, wr, chans, snr) if len(wt) > 1 else handle.ber_plan(s, wt[0], wr[0], chans, snr)
    name = plan.kernel
    plan.close()
    monkeypatch.delenv("WOFDM_DEBUG")
    m = re.findall(r"\[wofdm\] (\S+): smem \d+ B, (\d+) CTAs/SM", capfd.readouterr().err)
    nb = [int(b) for k, b in m if k == name]
    assert nb, (name, m)
    cl = int(re.search(r"_cl(\d+)", name).group(1)) if "_cl" in name else 1
    return name, nb[-1], cl


def say(capfd, msg):
    with capfd.disabled():                   # (capfd reads the residency report; what a row measured goes to the terminal)
        print(msg)


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def grid(frames, cap, cl):
    """ber_host.cu: plan_launch_impl -- CTAs of a launch of `frames` frames with `cap` resident CTAs"""
    return min(frames, max(cap // cl, 1)) * cl


def random_segments(rng, n_snr, E, calls):
    """[0, E) of every point cut at random places, the pieces shuffled and dealt to `calls` calls"""
    segs = []
    for k in range(n_snr):
        cuts = np.unique(np.concatenate([[0, E], rng.integers(1, E, size=6)]))
        segs += [(k, int(a), int(b - a)) for a, b in zip(cuts[:-1], cuts[1:])]
    order = rng.permutation(len(segs))
    return [[segs[i] for i in order[c::calls]] for c in range(calls)]


@pytest.mark.parametrize("row", list(ROWS))
def test_counters_depend_on_the_frame_alone(handle, row, monkeypatch, capfd):
    name, N, cp, ttx, trx, bits, L, nv, prec, env, kern, conv, guard, Cn, E = ROWS[row]
    set_env(monkeypatch, env)
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits, noise_norm=conv, constellation=conv, guard=guard)
    s = to_sys(p, prec)
    wins = [O.perturbed_windows(p, seed=N + k)[:2] for k in range(nv - 1)] + [(O.rc_window_tx(p), O.rc_window_rx(p))]
    wt, wr = [w[0] for w in wins], [w[1] for w in wins]
    chans = O.synth_channels(Cn, L, seed=N + L)
    snr = low_snr(bits)
    seed, variant = 4242, 3
    kernel, nb, cl = plan_residency(handle, s, wt, wr, chans, snr, monkeypatch, capfd)
    for k in kern:
        assert (k[1:] not in kernel) if k[0] == "!" else (k in kernel), (row, kernel)
    if "_b2" in kernel:
        assert nb >= 2, (kernel, nb)
    F = len(snr) * Cn * E
    decisions = F * nv * (p.S - 1) * int(np.count_nonzero(p.active))
    if prec == 0 and ("f32t" in kernel or "f32r" in kernel):
        assert decisions >= BIG, (row, decisions)

    multi = lambda **kw: handle.ber_run_multi(s, wt, wr, chans, snr, E, seed=seed, variant=variant, **kw)
    ref = multi()
    ser = ref["sym_err"] / ref["sym_tot"]
    say(capfd, f"\n{row}: {kernel}, {nb} CTA(s)/SM, {F} frames x {nv} pair(s) = {decisions:.3g} decisions per reassignment, SER {np.round(ser, 3).tolist()}")
    assert np.all(ser[:, 0] > ser[:, 1]) and np.all(ser > 0.01) and np.all(ser < 0.9), ser   # low SNR; SER falls with SNR
    diffs = {}

    def check(what, got, keys=("bit_err", "sym_err", "sym_tot", "bit_tot"), want=ref):
        d = {k: int(np.abs(np.asarray(got[k]) - np.asarray(want[k])).sum()) for k in keys}
        if any(d.values()):
            diffs[what] = d

    def summed(parts, keys=("bit_err", "sym_err", "sym_tot", "bit_tot")):
        return {k: sum(q[k] for q in parts) for k in keys}

    # 1. the same call again
    check("again", multi())
    # 2. one resident CTA per SM: other frames per CTA, other neighbours
    sms = sm_count()
    if grid(F, nb * sms, cl) != grid(F, sms, cl):
        monkeypatch.setenv("WOFDM_MAX_CTAS_PER_SM", "1")
        check("one CTA per SM", multi())
        monkeypatch.delenv("WOFDM_MAX_CTAS_PER_SM")
    else:
        assert nb == 1, (kernel, nb)
    # 3. shards summed
    for K in (2, 47):
        check(f"{K} shards", summed([multi(shard=(i, K)) for i in range(K)]))
    # 4. and 5. the resolved-counter twin of the production kernel; the first-generation tensor-core kernel has none (its
    #    resolved calls run the staged kernel, whose fp32 arithmetic is another)
    if "ber_f32t_" not in kernel:
        rng = np.random.default_rng(F)
        segs = random_segments(rng, len(snr), E, 3)
        check("segments", summed([handle.ber_run_segments(s, wt, wr, chans, snr, E, sg, seed=seed, variant=variant) for sg in segs]))
        kw = dict(seed=seed, variant=variant, by_subcarrier=True, by_channel=True)
        res = handle.ber_run_resolved(s, wt, wr, chans, snr, E, **kw)
        check("resolved, summed over channels and bins", {k: res[k].sum(axis=(-2, -1)) for k in ("bit_err", "sym_err", "sym_tot", "bit_tot")})
        K = 47
        parts = summed([handle.ber_run_resolved(s, wt, wr, chans, snr, E, shard=(i, K), **kw) for i in range(K)])
        check(f"resolved, {K} shards, cell by cell", parts, want=res)
    # 6. each window pair alone
    if nv > 1:
        for v in range(nv):
            one = handle.ber_run(s, wt[v], wr[v], chans, snr, E, seed=seed, variant=variant + v)
            check(f"pair {v} alone", {k: one[k] for k in ("bit_err", "sym_err")}, keys=("bit_err", "sym_err"),
                  want={k: ref[k][v] for k in ("bit_err", "sym_err")})
            check(f"pair {v} alone (totals)", one, keys=("bit_tot", "sym_tot"))
    # 7. a handle that splits the job over every visible device
    n = ctypes.c_int(0)
    assert W.capi.load().wofdm_device_count(ctypes.byref(n)) == 0
    if n.value >= 2:
        with W.Handle(None) as hall:
            check(f"{n.value} devices", hall.ber_run_multi(s, wt, wr, chans, snr, E, seed=seed, variant=variant))
    else:
        say(capfd, f"{row}: one visible device, the multi-device reassignment is skipped")
    report = "; ".join(f"{what}: {d}" for what, d in diffs.items())
    say(capfd, f"{row}: {'counters differ -- ' + report if diffs else 'every reassignment equal'}")
    assert not diffs, f"{row} ({kernel}, {decisions:.3g} decisions): |counter differences| {report}"


# kernel substrings, name, N, cp, tail_tx, tail_rx, bits, precision
ANCHORS = {
    "tconv2_n256": (["f32t2_n256"], "WOLA", 256, 16, 8, 10, 4, 0),
    "tconv2_n1024": (["f32t2_n1024", "_cl2"], "WOLA", 1024, 64, 32, 40, 6, 0),
    "fp64_n1024": (["f64_n1024"], "WOLA", 1024, 64, 32, 40, 6, 1),
}


@pytest.mark.parametrize("row", list(ANCHORS))
def test_oracle_anchor(handle, row, monkeypatch, capfd):
    """A long job (2 SNR points x 2048 channels x ensemble 1: every (SNR, channel) cell of the by-channel counters is one
    frame, at least 8 frames per CTA).  32 frames that their CTA decided last -- after state of earlier frames in shared and
    tensor memory -- replayed through the oracle on the exported draws: fp64 equal, fp32 within the boundary-flip budget."""
    kern, name, N, cp, ttx, trx, bits, prec = ANCHORS[row]
    set_env(monkeypatch, {})
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits, noise_norm=1, constellation=1)
    s = to_sys(p, prec)
    vt, vr, _, _ = O.perturbed_windows(p, seed=7)
    Cn, L, seed, variant = 2048, 21, 99, 5
    chans = O.synth_channels(Cn, L, seed=12)
    snr = low_snr(bits)
    kernel, nb, cl = plan_residency(handle, s, [vt], [vr], chans, snr, monkeypatch, capfd)
    for k in kern:
        assert k in kernel, (row, kernel)
    F = len(snr) * Cn
    nslots = grid(F, nb * sm_count(), cl) // cl                    # frames in flight: frame j runs on slot j mod nslots
    assert F >= 8 * nslots, (F, nslots)
    r = handle.ber_run_resolved(s, [vt], [vr], chans, snr, 1, seed=seed, variant=variant, by_subcarrier=False, by_channel=True)
    ref = handle.ber_run(s, vt, vr, chans, snr, 1, seed=seed, variant=variant)
    assert np.array_equal(r["sym_err"][0].sum(axis=(1, 2)), ref["sym_err"])
    ids = np.sort(np.random.default_rng(3).choice(np.arange(F - nslots, F), size=32, replace=False))   # each its CTA's last frame
    sym, nz = handle.ber_draws(s, L, seed, variant, ids)
    got_s, got_b, want_s, want_b, slack = [], [], [], [], 0
    for k, f in enumerate(ids):
        si, c = divmod(int(f), Cn)                                 # ensemble 1: frame f = si * C + c
        o = O.frame_chain_structured(p, vt, vr, chans[:, c], snr[si], sym[k].T, nz[k])
        want_s.append(o.sym_err)
        want_b.append(o.bit_err)
        got_s.append(int(r["sym_err"][0, si, c, 0]))
        got_b.append(int(r["bit_err"][0, si, c, 0]))
        slack += flip_budget(p, [o.eq])
    got_s, got_b, want_s, want_b = map(np.asarray, (got_s, got_b, want_s, want_b))
    say(capfd, f"\n{row}: {kernel}, {nslots} frames in flight, {F / nslots:.1f} frames per CTA, oracle {want_s.sum()} symbol errors "
          f"in 32 frames, device {got_s.sum()}, flip budget {slack}")
    assert want_s.sum() > 0
    if prec == 1:
        assert np.array_equal(got_s, want_s) and np.array_equal(got_b, want_b)
    else:
        assert np.abs(got_s - want_s).sum() <= slack, (got_s - want_s, slack)
        assert np.abs(got_b - want_b).sum() <= 3 * slack, (got_b - want_b, slack)
