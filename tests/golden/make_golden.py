"""Generate tests/golden/*.npz by executing the REFERENCE itself.

Run:  WOFDM_REFERENCE=<checkout of felipescoelho/w-ofdm-optimization> python -B tests/golden/make_golden.py
The reference is imported read-only (bytecode writing disabled); tests read only the committed .npz files.

What is stored
* ser_<sys>.npz     -- inputs + the SER vectors returned by the reference's own Monte-Carlo
                       loops (``wOFDMSystem.__run_sim_mc`` / ``__run_sim_cp_mc``, un-jitted
                       ``py_func`` under ``np.random.seed``), python/ofdm_utils/wofdm_simulation.py:85-366.
                       One of the cases per system is a single frame (1 SNR, 1 channel,
                       ensemble 1), so its SER pins that frame's symbol-error COUNT.
* interf_<sys>.npz  -- inputs + ``interf_power`` outputs (python/ofdm_utils/interf_calc.py:20-113)
                       on the mean of a stored channel set.
"""
import os
import sys
import tempfile

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.environ["WOFDM_REFERENCE"], "python"))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

from oracle import wofdm_oracle as O  # noqa: E402  (fixture inputs only: windows, channels)
from ofdm_utils.wofdm_simulation import wOFDMSystem  # noqa: E402
from ofdm_utils.transmitter import gen_rc_window_tx  # noqa: E402
from ofdm_utils.receiver import gen_rc_window_rx  # noqa: E402
from ofdm_utils.interf_calc import interf_power  # noqa: E402

MC = wOFDMSystem._wOFDMSystem__run_sim_mc.py_func
MC_CP = wOFDMSystem._wOFDMSystem__run_sim_cp_mc.py_func

N, CP = 256, 16


def tails(name):
    return (8 if name in ("CPW", "WOLA", "CPwtx", "wtx") else 0,
            10 if name in ("CPW", "WOLA", "CPwrx", "wrx") else 0)


def ref_mats(name, vt, vr, ttx, trx):
    s = wOFDMSystem(name, N, CP, ttx, trx, "/tmp/unused")
    if name == "CP":
        return s, s.add_red_mat @ s.idft_mat, s.dft_mat @ s.rm_red_mat, None, None
    tx = np.diag(vt) @ s.add_red_mat @ s.idft_mat
    tx_rc = gen_rc_window_tx(N, CP, s.cs_len, ttx) @ s.add_red_mat @ s.idft_mat
    rx = s.dft_mat @ s.circ_shift_mat @ s.overlap_add_mat @ np.diag(vr) @ s.rm_red_mat
    rx_rc = s.dft_mat @ s.circ_shift_mat @ s.overlap_add_mat @ gen_rc_window_rx(N, trx) @ s.rm_red_mat
    return s, tx, rx, tx_rc, rx_rc


def run_ser(name, S, channels, ensemble, snr, seed, vt, vr, ttx, trx):
    _, tx, rx, tx_rc, rx_rc = ref_mats(name, vt, vr, ttx, trx)
    np.random.seed(seed)
    if name == "CP":
        ser = MC_CP(tx, rx, S, channels, ensemble, snr)
        return np.stack([ser])
    a, b = MC(tx, tx_rc, rx, rx_rc, S, channels, ensemble, snr, ttx, True)
    return np.stack([a, b])


def main():
    chans = O.synth_channels(250, 21, seed=0)
    for name in O.SYSTEMS:
        ttx, trx = tails(name)
        p = O.system_params(name, N, CP, ttx, trx)
        vt, vr, xt, xr = O.perturbed_windows(p, seed=11)
        out = dict(name=name, N=N, cp=CP, tail_tx=ttx, tail_rx=trx, v_tx=vt, v_rx=vr, x_tx=xt, x_rx=xr)
        # case A: a small sweep (2 SNR x 2 channels x ensemble 2, S=4)
        out["A_S"] = 4
        out["A_channels"] = chans[:, :2]
        out["A_ensemble"] = 2
        out["A_snr"] = np.array([8.0, 24.0])
        out["A_seed"] = 7
        out["A_ser"] = run_ser(name, 4, chans[:, :2], 2, out["A_snr"], 7, vt, vr, ttx, trx)
        # case B: single frames (full S=16), one per SNR value, each its own seed
        snrs = np.array([0.0, 15.0, 30.0])
        out["B_S"] = 16
        out["B_channels"] = chans[:, 2:3]
        out["B_snr"] = snrs
        out["B_seed"] = np.array([21, 22, 23])
        out["B_ser"] = np.stack([run_ser(name, 16, chans[:, 2:3], 1, snrs[i:i + 1], 21 + i, vt, vr, ttx, trx)[:, 0]
                                 for i in range(3)])
        np.savez_compressed(os.path.join(HERE, f"ser_{name}.npz"), **out)
        print(name, "A", out["A_ser"].tolist(), "B", out["B_ser"].tolist())

    # interference: interf_power loads 'channels/vehicularA.npy' relative to the CWD (interf_calc.py:60,80)
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "channels"))
        np.save(os.path.join(td, "channels", "vehicularA.npy"), chans[:, :16])
        cwd = os.getcwd()
        os.chdir(td)
        try:
            for name in O.SYSTEMS:
                ttx, trx = tails(name)
                p = O.system_params(name, N, CP, ttx, trx)
                vt, vr, _, _ = O.perturbed_windows(p, seed=11)
                if name == "CP":
                    P = interf_power("CP", [None, None], N, CP, 0, 0)
                    res = dict(P_opt=P)
                else:
                    Po, Prc = interf_power(name, [np.diag(vt), np.diag(vr)], N, CP, ttx, trx)
                    res = dict(P_opt=Po, P_rc=Prc)
                np.savez_compressed(os.path.join(HERE, f"interf_{name}.npz"), name=name, N=N, cp=CP,
                                    tail_tx=ttx, tail_rx=trx, v_tx=vt, v_rx=vr,
                                    channels=chans[:, :16], **res)
                print(name, "interf total", float(np.sum(res["P_opt"])))
        finally:
            os.chdir(cwd)


if __name__ == "__main__":
    main()
