"""CPU: the oracle against the golden vectors produced by the reference itself
(tests/golden/make_golden.py).  Bit-exact: the SER vectors must be identical."""
import numpy as np
import pytest

from oracle import wofdm_oracle as O
from helpers import GOLDEN, golden_params, golden_windows, load_ser_golden, replay_frames


@pytest.mark.parametrize("name", O.SYSTEMS)
def test_ser_sweep_matches_reference(name):
    g = load_ser_golden(name)
    p = golden_params(g, g["A_S"])
    wins = golden_windows(g, p)
    np.random.seed(int(g["A_seed"]))
    ser = O.ser_sweep_replay(p, wins, g["A_channels"], int(g["A_ensemble"]), g["A_snr"], dense=True)
    assert np.array_equal(ser, g["A_ser"])


@pytest.mark.parametrize("name", O.SYSTEMS)
def test_single_frames_match_reference_counts(name):
    """Case B: one frame per SNR value -> the reference's SER pins the frame's error count,
    for the dense AND the structured form of the chain."""
    g = load_ser_golden(name)
    p = golden_params(g, g["B_S"])
    wins = golden_windows(g, p)
    for i, snr in enumerate(g["B_snr"]):
        fr = replay_frames(p, wins, g["B_channels"], 1, [snr], int(g["B_seed"][i]))[0]
        for w, (vt, vr) in enumerate(wins):
            want = g["B_ser"][i][w] * (p.N * (p.S - 1))
            assert abs(want - round(want)) < 1e-9
            for chain in (O.frame_chain_dense, O.frame_chain_structured):
                res = chain(p, vt, vr, fr["chan"], fr["snr"], fr["sym_idx"], fr["noise"][w])
                assert res.sym_err == int(round(want)), (name, snr, w, chain.__name__)


@pytest.mark.parametrize("name", ["WOLA", "CPwtx", "wrx"])
def test_replay_at_cp22_matches_stored_vectors(name):
    """np.random replayed at cp = 22, S = 3 (tests/golden/make_golden_replay.py): the dense AND the structured form must
    give the stored SER vectors bit for bit.  The stored file names its source: as committed it is the oracle's dense
    replay (the reference could not be run when it was made), so this pins the oracle against drift and the structured
    form against the dense one; regenerated from the reference it checks both against the reference."""
    g = np.load(f"{GOLDEN}/ser_replay.npz")
    ttx = 8 if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0
    trx = 10 if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0
    p = O.system_params(name, int(g["N"]), int(g["cp"]), ttx, trx, S=int(g["S"]))
    wins = [(g[f"{name}_v_tx"], g[f"{name}_v_rx"]), (O.rc_window_tx(p), O.rc_window_rx(p))]
    for dense in (True, False):
        np.random.seed(int(g[f"{name}_seed"]))
        ser = O.ser_sweep_replay(p, wins, g[f"{name}_channels"], int(g["ensemble"]), g["snr"], dense=dense)
        assert np.array_equal(ser, g[f"{name}_ser"]), (name, dense, str(g["source"]))


@pytest.mark.parametrize("name", O.SYSTEMS)
def test_structured_equals_dense(name):
    g = load_ser_golden(name)
    p = golden_params(g, 5)
    rng = np.random.default_rng(5)
    vt, vr = golden_windows(g, p)[0]
    h = g["B_channels"][:, 0]
    idx = rng.integers(0, 16, size=(p.N, p.S))
    nz = rng.standard_normal(O.noise_len(p, len(h))) + 1j * rng.standard_normal(O.noise_len(p, len(h)))
    a = O.frame_chain_dense(p, vt, vr, h, 20.0, idx, nz)
    b = O.frame_chain_structured(p, vt, vr, h, 20.0, idx, nz)
    assert np.abs(a.tx_stream - b.tx_stream).max() < 1e-13
    assert np.abs(a.Y - b.Y).max() < 1e-10 * np.abs(a.Y).max()
    assert np.linalg.norm(a.eq - b.eq) < 1e-10 * np.linalg.norm(a.eq)
    assert np.array_equal(a.dec_idx, b.dec_idx)


@pytest.mark.parametrize("name", O.SYSTEMS)
def test_interference_matches_reference(name):
    g = np.load(f"{GOLDEN}/interf_{name}.npz")
    ttx, trx = int(g["tail_tx"]), int(g["tail_rx"])
    if name == "CP":
        ttx = trx = 0
    p = O.system_params(name, int(g["N"]), int(g["cp"]), ttx, trx)
    h = g["channels"].mean(axis=1)
    vt, vr = (np.ones(p.n_tx), np.ones(p.N)) if name == "CP" else (g["v_tx"], g["v_rx"])
    P = O.interf_power_dense(p, vt, vr, h)
    assert np.allclose(P, g["P_opt"], rtol=1e-9, atol=1e-18)
    if name != "CP":
        Prc = O.interf_power_dense(p, O.rc_window_tx(p), O.rc_window_rx(p), h)
        assert np.allclose(Prc, g["P_rc"], rtol=1e-9, atol=1e-18)


@pytest.mark.parametrize("name", ["wtx", "WOLA", "CPW"])
def test_gram_form_equals_dense(name):
    g = np.load(f"{GOLDEN}/interf_{name}.npz")
    p = O.system_params(name, 64, 8, 4 if int(g["tail_tx"]) else 0, 4 if int(g["tail_rx"]) else 0)
    vt, vr, _, _ = O.perturbed_windows(p, seed=2)
    h = g["channels"][:, 3]
    a = O.interf_power_dense(p, vt, vr, h)
    b = O.interf_power_gram(p, vt, vr, h)
    assert np.allclose(a, b, rtol=1e-10, atol=1e-18)


def test_matlab_convention_tables():
    """Documented qammod(0:15,16) listing (SURVEY section 8c) and unit average power."""
    pts = O.qam_points(4, 1) * np.sqrt(10)
    want = np.array([-3 + 3j, -3 + 1j, -3 - 3j, -3 - 1j, -1 + 3j, -1 + 1j, -1 - 3j, -1 - 1j,
                     3 + 3j, 3 + 1j, 3 - 3j, 3 - 1j, 1 + 3j, 1 + 1j, 1 - 3j, 1 - 1j])
    assert np.allclose(pts, want)
    assert np.allclose(O.qam_points(2, 1) * np.sqrt(2), [-1 + 1j, -1 - 1j, 1 + 1j, 1 - 1j])
    for b in (2, 4, 6, 8):
        for conv in (0, 1):
            pts = O.qam_points(b, conv)
            assert np.array_equal(O.hard_decision(pts, b, conv), np.arange(1 << b))
            if conv == 1:
                assert abs(np.mean(np.abs(pts) ** 2) - 1) < 1e-12
            assert np.array_equal(O.hard_decision_argmin(pts * (1 + 1e-3), pts), np.arange(1 << b))


def test_decision_tie_rule_is_first_minimum():
    pts = O.qam_points(4, 0)
    x = np.array([0 + 0j, -2 - 2j, 2 + 2j, 0.0 + 3j, 5 + 5j, -7 - 0j])
    assert np.array_equal(O.hard_decision(x, 4, 0), O.hard_decision_argmin(x, pts))


@pytest.mark.parametrize("name,cp,guard,S", [("wtx", 16, 64, 16), ("WOLA", 22, 64, 5), ("CP", 10, 0, 3), ("CPW", 32, 100, 2)])
def test_mask_product_form_equals_the_filter_chain(name, cp, guard, S):
    """The algebra behind csrc/mask_gemm.cu: the DFT-domain mask of main_channel_mask.m:398-417 (mask_symbols, restated line
    by line) equals one constant matrix applied to the lattice points, with the filter tail of the previous symbol folded
    into the K dimension."""
    ttx = 8 if name in ("wtx", "WOLA", "CPW", "CPwtx") else 0
    trx = 10 if name in ("WOLA", "CPW", "wrx", "CPwrx") else 0
    p = O.system_params(name, 256, cp, ttx, trx, S=S, bits=4, noise_norm=1, constellation=1, guard=guard)
    v_tx, _, _, _ = O.perturbed_windows(p, seed=cp)
    rng = np.random.default_rng(cp)
    sym_idx = rng.integers(0, 16, size=(p.N, S))
    X = np.where(p.active[:, None], O.qam_points(p.bits, p.constellation)[sym_idx], 0.0)
    x = np.fft.ifft(X, axis=0)
    i = np.arange(p.n_tx)
    want = O.mask_symbols(v_tx[:, None] * x[(i - p.cp) % p.N, :], 10)
    nact = p.N - 2 * guard
    bins = (np.arange(nact) + guard + p.N // 2) % p.N
    got = O.mask_symbols_product(p, v_tx, X[bins, :], 10)
    assert got.shape == want.shape == (p.n_tx, S)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
