"""Statistical golden: SER curves produced by the REFERENCE's own jitted Monte-Carlo loops
(wOFDMSystem.__run_sim_mc / __run_sim_cp_mc, python/ofdm_utils/wofdm_simulation.py:85-366, numba as shipped) on
enough frames that a production run of the device kernel (its own Philox draws) can be required to fall inside
the reference's confidence interval at every SNR point (north star: "BER must fall within the 95 % CI of the
reference").  Stores the inputs, the reference's SER (optimised and RC windows) and the number of frames behind it.

Run:  WOFDM_REFERENCE=<checkout of felipescoelho/w-ofdm-optimization> python -B tests/golden/make_golden_stat.py   (~2 min)"""
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.environ["WOFDM_REFERENCE"], "python"))
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
from oracle import wofdm_oracle as O  # noqa: E402  (fixture inputs only)
from make_golden import ref_mats, tails, MC, MC_CP, N, CP  # noqa: E402
from ofdm_utils.wofdm_simulation import wOFDMSystem  # noqa: E402

MCJ = wOFDMSystem._wOFDMSystem__run_sim_mc          # the jitted loops, as the reference runs them
MCJ_CP = wOFDMSystem._wOFDMSystem__run_sim_cp_mc

chans = O.synth_channels(250, 21, seed=0)[:, 10:14]
snr = np.array([-5.0, 5.0, 15.0, 25.0, 40.0])
ENS, S = 150, 16
out = dict(channels=chans, snr=snr, ensemble=ENS, S=S, N=N, cp=CP)
for name in O.SYSTEMS:
    ttx, trx = tails(name)
    p = O.system_params(name, N, CP, ttx, trx)
    vt, vr, _, _ = O.perturbed_windows(p, seed=11)
    _, tx, rx, tx_rc, rx_rc = ref_mats(name, vt, vr, ttx, trx)
    if name == "CP":
        ser = np.stack([MCJ_CP(tx, rx, S, chans, ENS, snr)])
    else:
        a, b = MCJ(tx, tx_rc, rx, rx_rc, S, chans, ENS, snr, ttx, True)
        ser = np.stack([a, b])
    out[f"ser_{name}"] = ser
    out[f"vtx_{name}"] = vt
    out[f"vrx_{name}"] = vr
    print(name, np.round(ser, 4).tolist())
np.savez_compressed(os.path.join(HERE, "ser_statistical.npz"), **out)
