"""tests/golden/ser_replay.npz: the SER replay at a second cyclic-prefix length -- N = 256, cp = 22, S = 3, two channels x
ensemble 2 at 3 and 21 dB, optimised and RC windows -- for WOLA, CPwtx and wrx (seeds 101, 102, 103): draws the cp = 16
vectors of make_golden.py do not contain.

Run:  WOFDM_REFERENCE=<checkout of felipescoelho/w-ofdm-optimization> python -B tests/golden/make_golden_replay.py
      stores the SER vectors of the reference's own Monte-Carlo loop (wOFDMSystem.__run_sim_mc, un-jitted py_func
      under np.random.seed), source = "reference".
      python -B tests/golden/make_golden_replay.py --oracle
      stores the oracle's dense replay instead, source = "oracle".

The committed file was made with --oracle, because the reference could not be run when it was written.  It pins the
oracle's replay at cp = 22 against drift; it does not check it against the reference.  Regenerating it from the
reference restores that check with no change to tests/test_oracle_golden.py.
"""
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import numpy as np  # noqa: E402

from oracle import wofdm_oracle as O  # noqa: E402  (fixture inputs: windows, channels)

N, CP, S, ENSEMBLE = 256, 22, 3, 2
SNR = np.array([3.0, 21.0])
CASES = (("WOLA", 101), ("CPwtx", 102), ("wrx", 103))


def reference_ser(name, p, vt, vr, chans, seed):
    from ofdm_utils.wofdm_simulation import wOFDMSystem
    from ofdm_utils.transmitter import gen_rc_window_tx
    from ofdm_utils.receiver import gen_rc_window_rx
    s = wOFDMSystem(name, N, CP, p.tail_tx, p.tail_rx, "/tmp/unused")
    tx = np.diag(vt) @ s.add_red_mat @ s.idft_mat
    tx_rc = gen_rc_window_tx(N, CP, s.cs_len, p.tail_tx) @ s.add_red_mat @ s.idft_mat
    rx = s.dft_mat @ s.circ_shift_mat @ s.overlap_add_mat @ np.diag(vr) @ s.rm_red_mat
    rx_rc = s.dft_mat @ s.circ_shift_mat @ s.overlap_add_mat @ gen_rc_window_rx(N, p.tail_rx) @ s.rm_red_mat
    np.random.seed(seed)
    a, b = wOFDMSystem._wOFDMSystem__run_sim_mc.py_func(tx, tx_rc, rx, rx_rc, S, chans, ENSEMBLE, SNR, p.tail_tx, True)
    return np.stack([a, b])


def oracle_ser(name, p, vt, vr, chans, seed):
    np.random.seed(seed)
    return O.ser_sweep_replay(p, [(vt, vr), (O.rc_window_tx(p), O.rc_window_rx(p))], chans, ENSEMBLE, SNR, dense=True)


def main():
    if "--oracle" in sys.argv[1:]:
        source, ser = "oracle", oracle_ser
    else:
        sys.path.insert(0, os.path.join(os.environ["WOFDM_REFERENCE"], "python"))
        source, ser = "reference", reference_ser
    out = dict(source=source, N=N, cp=CP, S=S, ensemble=ENSEMBLE, snr=SNR, names=np.array([n for n, _ in CASES]))
    for name, seed in CASES:
        ttx = 8 if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0
        trx = 10 if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0
        p = O.system_params(name, N, CP, ttx, trx, S=S)
        vt, vr, _, _ = O.perturbed_windows(p, seed=seed)
        chans = O.synth_channels(2, 21, seed=seed)
        out.update({f"{name}_seed": seed, f"{name}_v_tx": vt, f"{name}_v_rx": vr, f"{name}_channels": chans,
                    f"{name}_ser": ser(name, p, vt, vr, chans, seed)})
        print(source, name, out[f"{name}_ser"].tolist())
    np.savez_compressed(os.path.join(HERE, "ser_replay.npz"), **out)


if __name__ == "__main__":
    main()
