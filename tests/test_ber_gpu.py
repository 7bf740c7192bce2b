"""GPU parity tests of K1 through the C-ABI (ctypes), against the oracle and the golden vectors.

Verify mode injects the reference's own draws (np.random replayed in the reference's call order):
  fp64: equalised symbols <= 1e-9 relative, decisions and error counts bit-exact;
  fp32: equalised symbols <= 1e-4 relative (frame norm), decisions bit-exact wherever the oracle's
        equalised symbol is farther than 1e-3 (lattice units) from a decision boundary.
"""
import numpy as np
import pytest

import wofdm_b200 as W
from oracle import wofdm_oracle as O
from helpers import golden_params, golden_windows, load_ser_golden, replay_frames

pytestmark = pytest.mark.gpu

TOL = {0: 1e-4, 1: 1e-9}
# fp32: largest deviation of ONE equalised symbol, relative to the frame's largest symbol (lattice units).  Observed over the
# whole suite on a B200: 4.7e-5 (a deep-fade bin; printed by test_zz_report_observed_fp32_slack), at most 1 decision per
# frame close enough to a boundary to differ legitimately, production counters equal to the oracle's in every replay.
# The north star allows 1e-4 on the frame norm; the per-symbol budget is the same number.
FP32_SYM_TOL = 1e-4
OBSERVED = {"unsafe": 0, "dev": 0.0, "prod": 0.0}


def flip_budget(p, eqs, tol=1e-4):
    """How many decisions fp32 rounding may flip: symbols whose oracle value lies within `tol` (relative to max(1, |x|),
    lattice units -- the north star's fp32 tolerance) of a decision boundary."""
    m = O.qam_levels(p.bits)
    sc = O.qam_scale(p.bits, p.constellation)
    n = 0
    for eq in eqs:
        x = eq[p.active] / sc
        n += int(np.count_nonzero(boundary_distance(x, m) <= tol * np.maximum(1.0, np.abs(x))))
    return n


@pytest.fixture(scope="module")
def handle():
    with W.Handle([0]) as h:
        yield h


def to_sys(p, precision):
    return W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift,
                  bits=p.bits, S=p.S, noise_norm=p.noise_norm, constellation=p.constellation, precision=precision,
                  guard=p.guard)


def boundary_distance(eq_lattice, m):
    """distance of each equalised symbol (lattice units) to the nearest decision boundary"""
    def ax(v):
        b = np.arange(-(m - 2), m - 1, 2.0)          # boundaries at even integers
        return np.min(np.abs(v[..., None] - b), axis=-1) if b.size else np.full(v.shape, np.inf)
    return np.minimum(ax(eq_lattice.real), ax(eq_lattice.imag))


def check_frames(handle, p, vt, vr, frames_in, precision, force_staged=False, direct=False, no_tconv=False):
    """frames_in: list of (chan, snr, sym_idx (N,S), noise)"""
    s = to_sys(p, precision)
    F = len(frames_in)
    chan = np.stack([f[0] for f in frames_in], axis=1)
    snr = np.array([f[1] for f in frames_in])
    sym = np.stack([f[2].T for f in frames_in])                      # (F, S, N)
    nz = np.stack([f[3] for f in frames_in])
    eq, dec, be, se = handle.ber_verify(s, vt, vr, chan, snr, sym, nz, force_staged=force_staged, direct=direct, no_tconv=no_tconv)
    m = O.qam_levels(p.bits)
    sc = O.qam_scale(p.bits, p.constellation)
    for i, (h, snr_i, idx, noise) in enumerate(frames_in):
        ref = O.frame_chain_structured(p, vt, vr, h, snr_i, idx, noise)
        got = eq[i].T                                                # (N, S-1)
        rel = np.linalg.norm(got - ref.eq) / np.linalg.norm(ref.eq)
        assert rel < TOL[precision], (i, rel)
        d = dec[i].T
        if precision == 1:
            assert np.array_equal(d, ref.dec_idx), i
            assert se[i] == ref.sym_err and be[i] == ref.bit_err, i
        else:
            # a decision may differ from the oracle's only where the device's OWN deviation (twice it, for the rounding of
            # the slicer's input) reaches a decision boundary; the deviation itself is bounded per symbol
            dev = np.abs(got - ref.eq) / sc
            assert dev.max() <= FP32_SYM_TOL * max(1.0, np.abs(ref.eq / sc).max()), (i, dev.max())
            safe = boundary_distance(ref.eq / sc, m) > 2.0 * dev + 1e-7
            safe |= ~p.active[:, None]          # null bins: exactly 0 + 0i on both sides, the tie rule decides
            assert np.array_equal(d[safe], ref.dec_idx[safe]), i
            assert abs(int(se[i]) - ref.sym_err) <= int((~safe).sum())
            OBSERVED["unsafe"] = max(OBSERVED["unsafe"], int((~safe).sum()))
            OBSERVED["dev"] = max(OBSERVED["dev"], float(dev.max() / max(1.0, np.abs(ref.eq / sc).max())))
        # counters are consistent with the returned decisions (over the sub-carriers that carry data)
        act = p.active
        assert se[i] == np.count_nonzero(d[act] != idx[act, 1:])
        assert be[i] == O.bit_errors(idx[act, 1:], d[act])


@pytest.mark.parametrize("precision", [1, 0])
@pytest.mark.parametrize("name", O.SYSTEMS)
def test_verify_against_reference_draws(handle, name, precision):
    """Golden case B: single frames drawn exactly as the reference draws them; the reference's own
    SER pins the symbol-error count of every frame."""
    g = load_ser_golden(name)
    p = golden_params(g, g["B_S"])
    wins = golden_windows(g, p)
    for i, snr in enumerate(g["B_snr"]):
        fr = replay_frames(p, wins, g["B_channels"], 1, [snr], int(g["B_seed"][i]))[0]
        for w, (vt, vr) in enumerate(wins):
            check_frames(handle, p, vt, vr, [(fr["chan"], fr["snr"], fr["sym_idx"], fr["noise"][w])], precision)
            if precision == 1:
                s = to_sys(p, 1)
                _, _, _, se = handle.ber_verify(s, vt, vr, fr["chan"][:, None], [fr["snr"]],
                                                fr["sym_idx"].T[None], fr["noise"][w][None])
                assert int(se[0]) == int(round(g["B_ser"][i][w] * p.N * (p.S - 1)))


@pytest.mark.parametrize("precision", [1, 0])
@pytest.mark.parametrize("N,S,bits,conv,nn", [(16, 3, 2, 0, 0), (32, 5, 4, 1, 1), (64, 16, 6, 1, 0), (128, 7, 8, 0, 1),
                                              (256, 16, 4, 1, 1), (256, 4, 4, 0, 0), (256, 9, 4, 1, 1), (512, 4, 6, 0, 0), (1024, 16, 6, 1, 0)])
def test_verify_shapes_and_conventions(handle, N, S, bits, conv, nn, precision):
    rng = np.random.default_rng(N + S)
    cp, ttx, trx = N // 16, N // 32, 2 * (N // 64) if N >= 64 else 0
    for name in ("WOLA", "CPW", "CP"):
        a, b = (0, 0) if name == "CP" else (ttx, trx)
        p = O.system_params(name, N, max(cp, a + b), a, b, S=S, bits=bits, noise_norm=nn, constellation=conv)
        vt, vr, _, _ = O.perturbed_windows(p, seed=N)
        L = 21 if N >= 64 else 5
        frames = []
        for k in range(3):
            h = O.synth_channels(1, L, seed=k)[:, 0]
            n = O.noise_len(p, L)
            frames.append((h, 5.0 + 12 * k, rng.integers(0, 1 << bits, size=(N, S)),
                           rng.standard_normal(n) + 1j * rng.standard_normal(n)))
        check_frames(handle, p, vt, vr, frames, precision)
        check_frames(handle, p, vt, vr, frames, precision, force_staged=True)
        if precision == 0:
            check_frames(handle, p, vt, vr, frames, precision, direct=True)      # direct-form convolution over the whole frame
            check_frames(handle, p, vt, vr, frames, precision, no_tconv=True)    # register policies incl. the circular interior


@pytest.mark.parametrize("policy", ["tconv", "regs"])
def test_production_replay_matches_oracle(handle, policy, monkeypatch):
    """Production mode: export the on-device Philox draws of some frames, replay them through the
    oracle and require the same error counts (fp64 exact; fp32 up to boundary flips).  fp32 runs the tensor-core
    convolution kernel (draw = stream position) or, with WOFDM_NO_TCONV, the register policies (blocks of 17)."""
    if policy == "regs":
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    g = load_ser_golden("WOLA")
    chans = np.concatenate([g["A_channels"], g["B_channels"]], axis=1)      # (21, 3)
    snr = np.array([6.0, 18.0])
    ens = 2
    for precision in (1, 0):
        for conv, nn in ((0, 0), (1, 1)):
            p = golden_params(g, 16, constellation=conv, noise_norm=nn)
            vt, vr = golden_windows(g, p)[0]
            s = to_sys(p, precision)
            if precision == 0:
                plan = handle.ber_plan(s, vt, vr, chans, snr)
                assert ("f32t" in plan.kernel) == (policy == "tconv"), plan.kernel
            res = handle.ber_run(s, vt, vr, chans, snr, ens, seed=1234, variant=1)
            F = len(snr) * chans.shape[1] * ens
            ids = np.arange(F)
            sym, nz = handle.ber_draws(s, chans.shape[0], 1234, 1, ids)
            assert sym.min() >= 0 and sym.max() < 16 and len(np.unique(sym)) == 16
            assert abs(np.mean(np.abs(nz) ** 2) - 2.0) < 0.05
            want_sym = np.zeros(len(snr), dtype=np.int64)
            want_bit = np.zeros(len(snr), dtype=np.int64)
            slack = np.zeros(len(snr), dtype=np.int64)
            for f in ids:
                e = f % ens
                c = (f // ens) % chans.shape[1]
                si = f // (ens * chans.shape[1])
                r = O.frame_chain_structured(p, vt, vr, chans[:, c], snr[si], sym[f].T, nz[f])
                want_sym[si] += r.sym_err
                want_bit[si] += r.bit_err
                slack[si] += flip_budget(p, [r.eq])
            assert np.array_equal(res["sym_tot"], np.full(len(snr), chans.shape[1] * ens * p.N * (p.S - 1)))
            assert np.array_equal(res["bit_tot"], res["sym_tot"] * p.bits)
            if precision == 1:
                assert np.array_equal(res["sym_err"], want_sym) and np.array_equal(res["bit_err"], want_bit)
            else:
                # fp32: only symbols within the fp32 tolerance of a decision boundary may flip (a flip moves one level:
                # one symbol error, at most two bit errors in the natural map, one in Gray)
                assert np.all(np.abs(res["sym_err"] - want_sym) <= slack), (res["sym_err"], want_sym, slack)
                assert np.all(np.abs(res["bit_err"] - want_bit) <= 2 * slack), (res["bit_err"], want_bit, slack)
                OBSERVED["prod"] = max(OBSERVED["prod"], float(np.max(np.abs(res["sym_err"] - want_sym) / np.maximum(slack, 1))))


@pytest.mark.parametrize("name,N,cp,bits,nv,precision", [("WOLA", 256, 16, 4, 7, 0), ("wtx", 256, 22, 4, 2, 0), ("CPW", 512, 32, 6, 3, 0),
                                                        ("WOLA", 1024, 64, 6, 2, 0), ("WOLA", 256, 16, 4, 3, 1), ("wrx", 64, 8, 2, 2, 0)])
def test_window_variants_in_one_launch(handle, name, N, cp, bits, nv, precision):
    """The reference evaluates several window pairs on every frame's symbols (optimised + RC, wofdm_simulation.py:183-236;
    RC + six optimisation steps for WOLA / CPW, main_BER_calculation.m:118-198).  wofdm_ber_run_multi does that in one
    call -- one launch where the tensor-core kernel applies (fp32, N >= 256), one launch per pair otherwise -- and pair v
    must get EXACTLY the counters of a single-pair run with variant v."""
    sc = N // 256 if N >= 256 else 1
    ttx = (8 * sc if N >= 256 else 2) if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0
    trx = (10 * sc if N >= 256 else 2) if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits, noise_norm=1, constellation=1)
    s = to_sys(p, precision)
    wins = []
    for v in range(nv):
        if v == 1:
            wins.append((O.rc_window_tx(p), O.rc_window_rx(p)))                    # flat windows
        elif v == 4:
            rng = np.random.default_rng(v)                                           # windows that are not flat
            wins.append((rng.uniform(0.5, 1.0, p.n_tx), rng.uniform(0.5, 1.0, p.N + p.tail_rx)))
        else:
            vt, vr, _, _ = O.perturbed_windows(p, seed=10 + v)
            wins.append((vt * (0.9 + 0.05 * v), vr))
    chan = O.synth_channels(3, 21 if N >= 64 else 5, seed=3)
    snr = np.array([4.0, 16.0, 28.0])
    ens = 5 if N <= 256 else 2
    multi = handle.ber_run_multi(s, [w[0] for w in wins], [w[1] for w in wins], chan, snr, ens, seed=99, variant=2)
    plan = handle.ber_plan_multi(s, [w[0] for w in wins], [w[1] for w in wins], chan, snr)
    assert plan.fused == (precision == 0 and N >= 256), plan.kernel
    plan.launch(ens, seed=99, variant=2)
    be, se = plan.read()
    plan.close()
    assert np.array_equal(be, multi["bit_err"]) and np.array_equal(se, multi["sym_err"])
    for v, (vt, vr) in enumerate(wins):
        one = handle.ber_run(s, vt, vr, chan, snr, ens, seed=99, variant=2 + v)
        assert np.array_equal(one["bit_err"], multi["bit_err"][v]) and np.array_equal(one["sym_err"], multi["sym_err"][v]), v
        assert np.array_equal(one["bit_tot"], multi["bit_tot"]) and np.array_equal(one["sym_tot"], multi["sym_tot"])
    # different windows, different counters; same symbols: shards add up
    assert not np.array_equal(multi["bit_err"][0], multi["bit_err"][1])
    parts = [handle.ber_run_multi(s, [w[0] for w in wins], [w[1] for w in wins], chan, snr, ens, seed=99, variant=2, shard=(i, 3))
             for i in range(3)]
    assert np.array_equal(sum(q["bit_err"] for q in parts), multi["bit_err"])


@pytest.mark.parametrize("policy", ["tconv", "regs"])
@pytest.mark.parametrize("name,nn", [("WOLA", 0), ("CPW", 1), ("CP", 1)])
def test_production_replay_cluster_kernel(handle, name, nn, policy, monkeypatch):
    """N = 1024 (one frame per 2-CTA cluster): the exported Philox draws, replayed through the oracle, give the
    production counters -- pins the noise numbering, the DSMEM tail / halo and the cluster-wide sums of both cluster
    kernels (tensor-core convolution; register policy behind WOFDM_NO_TCONV)."""
    if policy == "regs":
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    N, S, bits = 1024, 16, 6
    a, b = (0, 0) if name == "CP" else (32, 40)
    p = O.system_params(name, N, 64, a, b, S=S, bits=bits, noise_norm=nn, constellation=1)
    vt, vr, _, _ = O.perturbed_windows(p, seed=5)
    chans = O.synth_channels(2, 21, seed=11)
    snr = np.array([12.0, 30.0])
    ens = 2
    for precision in (0, 1):
        s = to_sys(p, precision)
        res = handle.ber_run(s, vt, vr, chans, snr, ens, seed=77, variant=0)
        F = len(snr) * chans.shape[1] * ens
        ids = np.arange(F)
        sym, nz = handle.ber_draws(s, chans.shape[0], 77, 0, ids)
        want_sym = np.zeros(len(snr), dtype=np.int64)
        want_bit = np.zeros(len(snr), dtype=np.int64)
        slack = np.zeros(len(snr), dtype=np.int64)
        for f in ids:
            c = (f // ens) % chans.shape[1]
            si = f // (ens * chans.shape[1])
            r = O.frame_chain_structured(p, vt, vr, chans[:, c], snr[si], sym[f].T, nz[f])
            want_sym[si] += r.sym_err
            want_bit[si] += r.bit_err
            slack[si] += flip_budget(p, [r.eq])
        if precision == 1:
            assert np.array_equal(res["sym_err"], want_sym) and np.array_equal(res["bit_err"], want_bit)
        else:
            assert np.all(np.abs(res["sym_err"] - want_sym) <= slack), (res["sym_err"], want_sym, slack)
            assert np.all(np.abs(res["bit_err"] - want_bit) <= 3 * slack), (res["bit_err"], want_bit, slack)
            OBSERVED["prod"] = max(OBSERVED["prod"], float(np.max(np.abs(res["sym_err"] - want_sym) / np.maximum(slack, 1))))


@pytest.mark.parametrize("precision", [1, 0])
def test_smallest_shapes_and_degenerate_jobs(handle, precision):
    """Edge cases of the domain: a two-symbol frame (pilot + one data symbol), a one-tap (flat) channel, one channel,
    one SNR point, ensemble 1, no windows at all (CP-OFDM) and windows with the shortest tails -- production counters
    replayed through the oracle from the exported draws."""
    for name, N, cp, ttx, trx, S, L, bits in (("CP", 256, 16, 0, 0, 2, 1, 4), ("WOLA", 256, 10, 2, 2, 2, 3, 2),
                                               ("CPW", 64, 8, 2, 2, 3, 1, 6), ("wtx", 16, 4, 2, 0, 2, 2, 2)):
        p = O.system_params(name, N, cp, ttx, trx, S=S, bits=bits, noise_norm=1, constellation=1)
        vt, vr = O.rc_window_tx(p), O.rc_window_rx(p)
        chan = O.synth_channels(1, max(L, 2), seed=9)[:L]
        s = to_sys(p, precision)
        res = handle.ber_run(s, vt, vr, chan, [17.0], 1, seed=8)
        sym, nz = handle.ber_draws(s, L, 8, 0, np.arange(1))
        r = O.frame_chain_structured(p, vt, vr, chan[:, 0], 17.0, sym[0].T, nz[0])
        assert res["sym_tot"][0] == N * (S - 1) and res["bit_tot"][0] == N * (S - 1) * bits
        tol = 0 if precision == 1 else 3
        assert abs(int(res["sym_err"][0]) - r.sym_err) <= tol and abs(int(res["bit_err"][0]) - r.bit_err) <= tol + 1


def test_invalid_arguments_are_rejected(handle):
    """Error behaviour of the boundary: negative WOFDM_E* codes surface as WofdmError, nothing is launched."""
    good = W.params_from_name("WOLA", 256, 16, 8, 10, bits=4, S=16)
    vt, vr = W.capi.rc_window_tx(good), W.capi.rc_window_rx(good)
    chan = O.synth_channels(2, 21, seed=1)
    before = handle.launches
    for field, value in (("N", 200), ("bits", 3), ("S", 1), ("tail_rx", 5), ("cp", -1), ("rm", 7), ("noise_norm", 2),
                         ("constellation", 3), ("precision", 2), ("shift", 256)):
        bad = W.SysT(**{f: getattr(good, f) for f, _ in good._fields_})
        setattr(bad, field, value)
        with pytest.raises(W.WofdmError):
            handle.ber_run(bad, vt, vr, chan, [10.0], 1, seed=0)
    with pytest.raises(W.WofdmError):
        handle.ber_run(good, vt, vr, chan, [10.0], 0, seed=0)            # ensemble must be >= 1
    with pytest.raises(W.WofdmError):
        handle.ber_run(good, vt, vr, chan, [10.0], 1, seed=0, shard=(3, 2))
    with pytest.raises(W.WofdmError):
        handle.interf_power(good, vt, vr, chan, mode=5)
    with pytest.raises(W.WofdmError):
        W.params_from_name("OFDMA", 256, 16, 8, 10)
    assert handle.launches == before


def test_full_size_properties_configs1(handle):
    """BASELINE configs[1] at its full size (250 channels x 30 SNR points x ensemble 27 = 202 500 frames, 1e8 bits per
    point), checked through size-independent properties: exact totals, shard additivity, BER ~ 1/2 at -20 dB,
    monotone in SNR up to its Monte-Carlo error, the error floor of the interference-limited regime at +50 dB."""
    s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1)
    x_tx = np.concatenate([[1.0], np.clip(W.capi.rc_window_tx(s)[-8:] * (1 + 0.1 * np.random.default_rng(7).uniform(-1, 1, 8)), 0, 1)])
    vt, vr = W.capi.expand_window_tx(s, x_tx), W.capi.rc_window_rx(s)
    chan = O.synth_channels(250, 21, seed=1)
    snr = np.linspace(-20, 50, 30)
    full = handle.ber_run(s, vt, vr, chan, snr, 27, seed=2024)
    assert np.all(full["bit_tot"] == 250 * 27 * 256 * 4 * 15) and np.all(full["sym_tot"] == 250 * 27 * 256 * 15)
    parts = [handle.ber_run(s, vt, vr, chan, snr, 27, seed=2024, shard=(i, 2)) for i in range(2)]
    for k in full:
        assert np.array_equal(full[k], parts[0][k] + parts[1][k]), k
    ber = full["bit_err"] / full["bit_tot"]
    assert abs(ber[0] - 0.5) < 0.01
    se = np.sqrt(ber * (1 - ber) / (250 * 27 * 15))              # per-frame granularity: a conservative standard error
    assert np.all(np.diff(ber) <= 4 * (se[1:] + se[:-1]))
    assert 0 < ber[-1] < 0.05 and ber[-1] < ber[10]
    # symbol errors dominate bit errors, and a wrong symbol has 1..4 wrong bits
    assert np.all(full["sym_err"] <= full["bit_err"]) and np.all(full["bit_err"] <= 4 * full["sym_err"])


def test_tensor_core_convolution_is_fp32_grade(handle):
    """The tensor-core convolution (split fp16 stream x split fp16 taps, fp32 accumulation) against the register
    direct form on the same injected draws: the equalised symbols of the two fp32 kernels differ by rounding only
    (both sit ~1e-6 from the fp64 oracle), decisions identical away from decision boundaries; BASELINE configs[1]
    dispatches to it."""
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1)
    vt, vr, _, _ = O.perturbed_windows(p, seed=3)
    s = to_sys(p, 0)
    rng = np.random.default_rng(3)
    F = 6
    chan = O.synth_channels(F, 21, seed=9)
    n = O.noise_len(p, 21)
    snr = np.linspace(0.0, 50.0, F)
    sym = rng.integers(0, 16, size=(F, 16, 256))
    nz = rng.standard_normal((F, n)) + 1j * rng.standard_normal((F, n))
    plan = handle.ber_plan(s, vt, vr, chan, snr)
    assert "f32t" in plan.kernel, plan.kernel
    eq_t, dec_t, _, _ = handle.ber_verify(s, vt, vr, chan, snr, sym, nz)
    eq_d, dec_d, _, _ = handle.ber_verify(s, vt, vr, chan, snr, sym, nz, direct=True)
    for f in range(F):
        ref = O.frame_chain_structured(p, vt, vr, chan[:, f], snr[f], sym[f].T, nz[f]).eq.T
        e_t = np.linalg.norm(eq_t[f] - ref) / np.linalg.norm(ref)
        e_d = np.linalg.norm(eq_d[f] - ref) / np.linalg.norm(ref)
        assert e_t < 1e-5 and e_d < 1e-5, (f, e_t, e_d)            # north star: 1e-4 for fp32
        assert e_t < 4 * e_d + 1e-6, (f, e_t, e_d)
    assert np.mean(dec_t != dec_d) < 2e-3


@pytest.mark.parametrize("hscale,wscale", [(1e-6, 1.0), (1e4, 1.0), (1.0, 3e4), (3e-7, 1e-5)])
def test_tensor_core_kernel_is_scale_invariant(handle, hscale, wscale):
    """The tensor-core kernels stage the stream and the taps as fp16 pairs behind fixed scales; the host gives them a
    known range (unit-peak Tx window and taps, ber_host.cu: build_tables / cast_chan), which the chain allows: a common
    factor of the Tx signal or of a channel's taps cancels in the measured-power noise gain and the pilot equaliser.
    Channels in path-loss units or an un-normalised window must give the oracle's answer (ADVICE round 1)."""
    p = O.system_params("WOLA", 256, 16, 8, 10, S=16, bits=4, noise_norm=0, constellation=0)
    vt, vr, _, _ = O.perturbed_windows(p, seed=5)
    rng = np.random.default_rng(17)
    frames = []
    for k in range(3):
        h = O.synth_channels(1, 21, seed=40 + k)[:, 0] * hscale * (1.0 + k)
        n = O.noise_len(p, 21)
        frames.append((h, 10.0 + 15 * k, rng.integers(0, 16, size=(256, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n)))
    s = to_sys(p, 0)
    plan = handle.ber_plan(s, vt * wscale, vr, np.stack([f[0] for f in frames], axis=1), [10.0])
    assert "f32t" in plan.kernel, plan.kernel
    plan.close()
    check_frames(handle, p, vt * wscale, vr, frames, 0)
    # production mode: same counters as the well-scaled job, up to boundary flips (fp32 rounding differs with the scale)
    chan = O.synth_channels(4, 21, seed=50)
    snr = np.array([5.0, 25.0])
    a = handle.ber_run(s, vt, vr, chan, snr, 3, seed=9)
    b = handle.ber_run(s, vt * wscale, vr, chan * hscale, snr, 3, seed=9)
    assert np.all(np.abs(a["sym_err"] - b["sym_err"]) <= 3 + 0.002 * a["sym_err"]), (a["sym_err"], b["sym_err"])


def test_production_replay_frame_received_in_two_passes(handle):
    """S = 17 > 16 transforms per CTA: the register kernels receive the frame in two passes and the second one reads the
    stream after the pilot barriers, so the frame keeps its closing barrier (ADVICE round 1: WOLA, cp = 16 has rm = 6 <
    tail_tx = 8, where a missing barrier lets the next frame's first Tx tail land in the samples pass 2 still reads).
    Production counters of a job with several frames per CTA must equal the verify-mode kernel's (which always had the
    barrier) on the exported draws of every frame, exactly: same arithmetic, same code."""
    g = load_ser_golden("WOLA")
    chans = np.concatenate([g["A_channels"], g["B_channels"]], axis=1)
    snr = np.array([8.0, 30.0])
    ens = 200                                  # 1200 frames on <= 296 resident CTAs
    p = golden_params(g, 17, constellation=0, noise_norm=0)
    vt, vr = golden_windows(g, p)[0]
    s = to_sys(p, 0)
    plan = handle.ber_plan(s, vt, vr, chans, snr)
    assert "f32t" not in plan.kernel and "_c" in plan.kernel, plan.kernel       # a register-policy kernel
    plan.close()
    res = handle.ber_run(s, vt, vr, chans, snr, ens, seed=77)
    C = chans.shape[1]
    F = len(snr) * C * ens
    ids = np.arange(F)
    want_s, want_b = np.zeros(len(snr), dtype=np.int64), np.zeros(len(snr), dtype=np.int64)
    for lo in range(0, F, 300):
        part = ids[lo:lo + 300]
        sym, nz = handle.ber_draws(s, chans.shape[0], 77, 0, part)
        _, _, be, se = handle.ber_verify(s, vt, vr, chans[:, (part // ens) % C], snr[part // (ens * C)], sym, nz)
        np.add.at(want_s, part // (ens * C), se)
        np.add.at(want_b, part // (ens * C), be)
    assert np.array_equal(res["sym_err"], want_s) and np.array_equal(res["bit_err"], want_b)
    # and the oracle on a sample of the frames
    sym, nz = handle.ber_draws(s, chans.shape[0], 77, 0, ids[::97])
    _, _, _, se = handle.ber_verify(s, vt, vr, chans[:, (ids[::97] // ens) % C], snr[ids[::97] // (ens * C)], sym, nz)
    tot = sum(O.frame_chain_structured(p, vt, vr, chans[:, (f // ens) % C], snr[f // (ens * C)], sym[k].T, nz[k]).sym_err
              for k, f in enumerate(ids[::97]))
    assert abs(int(se.sum()) - tot) <= 3 + 0.002 * tot


@pytest.mark.parametrize("name,cp", [("WOLA", 16), ("CPwtx", 22), ("CPW", 10)])
def test_tensor_core_kernel_with_windows_that_are_not_flat(handle, name, cp):
    """The tensor-core kernel folds a flat Tx window into its constellation table and divides a flat Rx window out
    (every window the reference produces is flat between its tails); arbitrary windows take its general path."""
    ttx = 8 if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0
    trx = 10 if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0
    p = O.system_params(name, 256, cp, ttx, trx, S=16, bits=6, noise_norm=1, constellation=1)
    rng = np.random.default_rng(cp)
    vt = rng.uniform(0.5, 1.0, p.n_tx)
    vr = rng.uniform(0.5, 1.0, p.N + p.tail_rx)
    frames = []
    for k in range(2):
        h = O.synth_channels(1, 21, seed=30 + k)[:, 0]
        n = O.noise_len(p, 21)
        frames.append((h, 14.0 + 20 * k, rng.integers(0, 64, size=(256, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n)))
    check_frames(handle, p, vt, vr, frames, 0)
    check_frames(handle, p, vt, vr, frames, 0, direct=True)


@pytest.mark.parametrize("cp", [10, 22, 32])
@pytest.mark.parametrize("name", O.SYSTEMS)
def test_verify_every_system_over_the_cp_range(handle, name, cp):
    """settingsData's CP range (10..32) for all seven systems at N = 256, fp32, both channel policies: exercises the
    prefix / suffix copies of the circular-interior kernel (cp > tail_tx + L - 1, cs > tail_tx) and the outer-row
    logic of the direct kernels, which the CP = 16 goldens do not reach."""
    ttx = 8 if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0
    trx = 10 if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0
    p = O.system_params(name, 256, cp, ttx, trx, S=16, bits=4, noise_norm=cp % 4 == 0, constellation=1)
    vt, vr, _, _ = O.perturbed_windows(p, seed=cp)
    rng = np.random.default_rng(cp)
    frames = []
    for k in range(2):
        h = O.synth_channels(1, 21, seed=cp + k)[:, 0]
        n = O.noise_len(p, 21)
        frames.append((h, 8.0 + 15 * k, rng.integers(0, 16, size=(256, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n)))
    check_frames(handle, p, vt, vr, frames, 0)                       # tensor-core convolution (the production choice)
    check_frames(handle, p, vt, vr, frames, 0, direct=True)
    check_frames(handle, p, vt, vr, frames, 0, no_tconv=True)


@pytest.mark.parametrize("policy", ["tconv", "regs"])
@pytest.mark.parametrize("name,cp", [("WOLA", 40), ("CPW", 128), ("CPwtx", 96), ("wrx", 72), ("CP", 128)])
def test_verify_cluster_kernel_over_shapes(handle, name, cp, policy, monkeypatch):
    """N = 1024 (2-CTA cluster kernels: tensor-core convolution, and the register policy behind WOFDM_NO_TCONV), 4x scaled
    tails, other CP lengths than the stress configuration's 64."""
    if policy == "regs":
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    ttx = 32 if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0
    trx = 40 if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0
    p = O.system_params(name, 1024, cp, ttx, trx, S=16, bits=6, noise_norm=1, constellation=1)
    vt, vr, _, _ = O.perturbed_windows(p, seed=cp)
    rng = np.random.default_rng(cp)
    h = O.synth_channels(1, 21, seed=cp)[:, 0]
    n = O.noise_len(p, 21)
    frames = [(h, 22.0, rng.integers(0, 64, size=(1024, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n))]
    check_frames(handle, p, vt, vr, frames, 0)
    s = to_sys(p, 0)
    plan = handle.ber_plan(s, vt, vr, h[:, None], [22.0])
    assert "_cl" in plan.kernel and ("f32t" in plan.kernel) == (policy == "tconv"), plan.kernel
    plan.close()


@pytest.mark.parametrize("policy", ["tconv", "regs"])
@pytest.mark.parametrize("name", ["WOLA", "CPW", "CP"])
def test_verify_and_replay_n512_tuned_kernel(handle, name, policy, monkeypatch):
    """N = 512: one 512-thread CTA per frame (tensor-core convolution; register-resident policy with WOFDM_NO_TCONV),
    verify mode and a production replay."""
    if policy == "regs":
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    ttx, trx = (0, 0) if name == "CP" else (16, 20)
    p = O.system_params(name, 512, 32, ttx, trx, S=16, bits=4, noise_norm=1, constellation=1)
    vt, vr, _, _ = O.perturbed_windows(p, seed=3)
    rng = np.random.default_rng(5)
    h = O.synth_channels(2, 21, seed=6)
    n = O.noise_len(p, 21)
    frames = [(h[:, k], 12.0 + 10 * k, rng.integers(0, 16, size=(512, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n))
              for k in range(2)]
    check_frames(handle, p, vt, vr, frames, 0, no_tconv=(policy == "regs"))
    s = to_sys(p, 0)
    plan = handle.ber_plan(s, vt, vr, h, [20.0])
    assert "n512_t512" in plan.kernel and ("f32t" in plan.kernel) == (policy == "tconv"), plan.kernel
    plan.close()
    res = handle.ber_run(s, vt, vr, h, [20.0], 2, seed=31)
    sym, nz = handle.ber_draws(s, 21, 31, 0, np.arange(4))
    want = sum(O.frame_chain_structured(p, vt, vr, h[:, f // 2], 20.0, sym[f].T, nz[f]).sym_err for f in range(4))
    assert abs(int(res["sym_err"][0]) - want) <= 3


@pytest.mark.parametrize("policy", ["tconv", "regs"])
def test_device_draws_are_gaussian_and_uniform(handle, policy, monkeypatch):
    """Quality of the on-device draws (Philox4x32-10 + Box-Muller on the MUFU approximations, exported with
    wofdm_ber_draws): moments, Kolmogorov-Smirnov distance, independence of the two parts and of neighbours, uniform
    constellation indices -- for the fp32 kernels' numberings (draw = position / blocks of 17) and the fp64 one."""
    from scipy import stats
    if policy == "regs":
        monkeypatch.setenv("WOFDM_NO_TCONV", "1")
    else:
        monkeypatch.delenv("WOFDM_NO_TCONV", raising=False)
    s0 = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16)
    for precision in ((0, 1) if policy == "tconv" else (0,)):
        s = W.SysT(**{f: getattr(s0, f) for f, _ in s0._fields_})
        s.precision = precision
        sym, nz = handle.ber_draws(s, 21, 99, 0, np.arange(3000, 3024))
        z = nz.ravel()
        n = z.size                                            # ~1e5 complex samples
        for part in (z.real, z.imag):
            assert abs(part.mean()) < 4 / np.sqrt(n)
            assert abs(part.var() - 1) < 4 * np.sqrt(2 / n)
            assert abs(stats.kurtosis(part, fisher=False) - 3) < 4 * np.sqrt(24 / n)
            assert abs(stats.skew(part)) < 4 * np.sqrt(6 / n)
            assert stats.kstest(part, "norm").statistic < 1.95 / np.sqrt(n)      # 0.1 % level
            assert abs(np.corrcoef(part[:-1], part[1:])[0, 1]) < 4 / np.sqrt(n)
        assert abs(np.corrcoef(z.real, z.imag)[0, 1]) < 4 / np.sqrt(n)
        assert np.abs(z).max() > 4.0                          # the tails are there (32-bit radius uniform)
        counts = np.bincount(sym.ravel(), minlength=16)
        assert stats.chisquare(counts).pvalue > 1e-4
        # frames and variants are different streams
        _, nz_b = handle.ber_draws(s, 21, 99, 1, np.arange(3000, 3002))
        assert abs(np.corrcoef(nz[0].real, nz_b[0].real)[0, 1]) < 0.1 and not np.array_equal(nz[0], nz[1])


@pytest.mark.parametrize("precision", [1, 0])
@pytest.mark.parametrize("name,N,cp,ttx,trx,bits,guard", [("wtx", 256, 16, 8, 0, 4, 64), ("CPW", 256, 22, 8, 10, 4, 64),
                                                          ("WOLA", 256, 16, 8, 10, 6, 31), ("WOLA", 1024, 64, 32, 40, 6, 256),
                                                          ("CP", 512, 32, 0, 0, 2, 128), ("wrx", 64, 8, 0, 4, 4, 16)])
def test_guard_band(handle, name, N, cp, ttx, trx, bits, guard, precision):
    """Null sub-carriers on both sides of the centred spectrum (matlab/main_channel_mask.m:55,388-391: offset = N/4,
    zeros + ifftshift): verify mode against the oracle for every policy (exact fit, circular interior, cluster, N = 512,
    staged), and a production replay; only the N - 2*guard active bins are counted."""
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=bits, noise_norm=1, constellation=1, guard=guard)
    vt, vr, _, _ = O.perturbed_windows(p, seed=guard)
    rng = np.random.default_rng(guard + N)
    h = O.synth_channels(2, 21, seed=guard)
    n = O.noise_len(p, 21)
    frames = [(h[:, k], 10.0 + 12 * k, rng.integers(0, 1 << bits, size=(N, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n))
              for k in range(2)]
    check_frames(handle, p, vt, vr, frames, precision)
    if precision == 0:
        check_frames(handle, p, vt, vr, frames, precision, direct=True)
        check_frames(handle, p, vt, vr, frames, precision, no_tconv=True)
        check_frames(handle, p, vt, vr, frames, precision, force_staged=True)
    s = to_sys(p, precision)
    res = handle.ber_run(s, vt, vr, h, [18.0], 2, seed=guard)
    assert res["sym_tot"][0] == 4 * (N - 2 * guard) * 15 and res["bit_tot"][0] == res["sym_tot"][0] * bits
    sym, nz = handle.ber_draws(s, 21, guard, 0, np.arange(4))
    want_s = want_b = 0
    for f in range(4):
        r = O.frame_chain_structured(p, vt, vr, h[:, f // 2], 18.0, sym[f].T, nz[f])
        want_s += r.sym_err
        want_b += r.bit_err
    tol = 0 if precision == 1 else 3
    assert abs(int(res["sym_err"][0]) - want_s) <= tol and abs(int(res["bit_err"][0]) - want_b) <= tol + 2
    with pytest.raises(W.WofdmError):
        handle.ber_run(W.params_from_name(name, N, cp, ttx, trx, bits=8, guard=guard), vt, vr, h, [18.0], 1)


@pytest.mark.parametrize("name,N,cp,nn", [("WOLA", 256, 16, 0), ("CPW", 256, 32, 1), ("WOLA", 1024, 64, 1), ("CP", 1024, 128, 0)])
def test_long_channel_on_the_tensor_core_kernel(handle, name, N, cp, nn):
    """BASELINE configs[4]: "L = 21 (optionally 84)".  Channels of up to 84 taps stay on the tensor-core kernel (84 samples of
    convolution history in the Hankel operand, 22 MMAs per tile): verify mode against the oracle, production replay."""
    sc = N // 256
    ttx, trx = (0, 0) if name == "CP" else (8 * sc, 10 * sc)
    L = 84
    p = O.system_params(name, N, cp, ttx, trx, S=16, bits=4 if N == 256 else 6, noise_norm=nn, constellation=nn)
    vt, vr, _, _ = O.perturbed_windows(p, seed=N + cp)
    rng = np.random.default_rng(L + N)
    frames = []
    for k in range(2):
        h = O.synth_channels(1, L, seed=60 + k)[:, 0]
        n = O.noise_len(p, L)
        frames.append((h, 12.0 + 15 * k, rng.integers(0, 1 << p.bits, size=(N, 16)), rng.standard_normal(n) + 1j * rng.standard_normal(n)))
    check_frames(handle, p, vt, vr, frames, 0)
    s = to_sys(p, 0)
    chans = O.synth_channels(2, L, seed=70)
    snr = np.array([10.0, 26.0])
    plan = handle.ber_plan(s, vt, vr, chans, snr)
    assert "f32t2" in plan.kernel and "_l84" in plan.kernel, plan.kernel
    plan.close()
    ens = 2
    res = handle.ber_run(s, vt, vr, chans, snr, ens, seed=31)
    F = len(snr) * 2 * ens
    sym, nz = handle.ber_draws(s, L, 31, 0, np.arange(F))
    want, slack = np.zeros(2, dtype=np.int64), np.zeros(2, dtype=np.int64)
    for f in range(F):
        r = O.frame_chain_structured(p, vt, vr, chans[:, (f // ens) % 2], snr[f // (ens * 2)], sym[f].T, nz[f])
        want[f // (ens * 2)] += r.sym_err
        slack[f // (ens * 2)] += flip_budget(p, [r.eq])
    assert np.all(np.abs(res["sym_err"] - want) <= slack), (res["sym_err"], want, slack)


@pytest.mark.parametrize("which", ["n256", "multi", "n512", "n1024"])
def test_relaxed_barriers_against_debug_build(which):
    """The tensor-core kernel drops the barrier at the end of a frame, lets only the MMA-issuing warps wait for the stream
    (bar.arrive / bar.sync) and reuses its shared-memory buffers from frame to frame.  compute-sanitizer is closed on this
    GPU pool (profiles/r2_racecheck_attempt.txt), so the check is a second build of the library, libwofdm_dbg.so, in which
    all of that is a full CTA / cluster barrier (ber_tconv2.cuh: TCV2_DEBUG_BARRIERS): jobs with several frames per CTA
    (tools/sanitize_k1.py) must give bit-identical counters in both builds, run after run."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dbg = os.path.join(root, "w-ofdm-optimization_b200", "libwofdm_dbg.so")
    assert os.path.exists(dbg), "libwofdm_dbg.so is built by `make -C w-ofdm-optimization_b200/csrc` (__graft_entry__.build)"
    outs = []
    for lib in (None, dbg, None):
        env = dict(os.environ)
        env.pop("WOFDM_LIB", None)
        if lib:
            env["WOFDM_LIB"] = lib
        r = subprocess.run([sys.executable, os.path.join(root, "tools", "sanitize_k1.py"), which], env=env, capture_output=True,
                           text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append([l for l in r.stdout.splitlines() if l.startswith("COUNTERS")])
    assert outs[0] and outs[0] == outs[1] == outs[2], outs


def test_in_process_multi_device_handle_matches_one_device():
    """wofdm_create(&h, 0): ONE process that owns every visible GPU and splits each job's frames over them itself (this is
    the MEX gateway's handle; ber_host.cu: wofdm_ber_run_multi's sub-shards).  Counters must be identical to the one-device
    run -- draws depend on the global frame id only.  Needs >= 2 devices (the driver's multi-GPU box; skipped on one)."""
    import ctypes
    n = ctypes.c_int(0)
    assert W.capi.load().wofdm_device_count(ctypes.byref(n)) == 0
    if n.value < 2:
        pytest.skip("one visible device")
    p = O.system_params("WOLA", 256, 16, 8, 10, S=16, bits=4, noise_norm=0, constellation=0)
    vt, vr, _, _ = O.perturbed_windows(p, seed=2)
    chan = O.synth_channels(7, 21, seed=4)
    snr = np.array([3.0, 15.0, 27.0])
    with W.Handle([0]) as h1, W.Handle(None) as hall:
        for precision in (0, 1):
            s = to_sys(p, precision)
            a = h1.ber_run(s, vt, vr, chan, snr, 11, seed=5)
            b = hall.ber_run(s, vt, vr, chan, snr, 11, seed=5)
            for k in a:
                assert np.array_equal(a[k], b[k]), (precision, k)
        s = to_sys(p, 0)
        wins_t, wins_r = [vt, O.rc_window_tx(p)], [vr, O.rc_window_rx(p)]
        a = h1.ber_run_multi(s, wins_t, wins_r, chan, snr, 11, seed=6)
        b = hall.ber_run_multi(s, wins_t, wins_r, chan, snr, 11, seed=6)
        for k in a:
            assert np.array_equal(a[k], b[k]), k
        # the channel-mask chain: contiguous frame ranges per device, its mask product and K1 on each of them
        sg = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1, guard=64)
        wt, wr = W.capi.rc_window_tx(sg), W.capi.rc_window_rx(sg)
        a = h1.ber_run_masked(sg, wt, wr, chan, snr, 37, seed=7, variant=1)
        b = hall.ber_run_masked(sg, wt, wr, chan, snr, 37, seed=7, variant=1)
        for k in a:
            assert np.array_equal(a[k], b[k]), k
        # the interference path of a multi-device handle runs on its first device
        Pa = h1.interf_power(to_sys(p, 1), vt, vr, chan)
        Pb = hall.interf_power(to_sys(p, 1), vt, vr, chan)
        assert np.allclose(Pa, Pb, rtol=1e-12, atol=0)         # (row sums meet in atomicAdd(double): order-dependent rounding)


def test_zz_report_observed_fp32_slack():
    """Not a check of its own: prints what the fp32 parity tests above actually needed, so that their budgets stay honest
    (run with -s to see it; the asserts keep a regression from hiding inside the budgets)."""
    print(f"\nfp32 parity, observed over this run: most decisions of one frame that could legitimately differ = {OBSERVED['unsafe']}, "
          f"largest per-symbol deviation = {OBSERVED['dev']:.2e} (budget {FP32_SYM_TOL:.0e}), "
          f"largest production |counter - oracle| / flip budget = {OBSERVED['prod']:.2f}")
    assert OBSERVED["dev"] <= FP32_SYM_TOL
