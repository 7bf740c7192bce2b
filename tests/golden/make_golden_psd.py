"""Golden vectors for the PSD / out-of-band-radiation estimate (SURVEY 8f-3), produced by executing the REFERENCE's
wOFDMSystem.estimate_obr (python/ofdm_utils/timefreq_simulation.py:216-296) under np.random.seed; the symbols it drew
are recovered by replaying the same seed (its first and only RNG call is np.random.choice(symbols, (N - 96, 256))).

Run:  WOFDM_REFERENCE=<checkout of felipescoelho/w-ofdm-optimization> python -B tests/golden/make_golden_psd.py"""
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.environ["WOFDM_REFERENCE"], "python"))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import numpy as np  # noqa: E402
from ofdm_utils.timefreq_simulation import wOFDMSystem  # noqa: E402
from oracle import wofdm_oracle as O  # noqa: E402  (windows only: the fixtures' optimised-window stand-ins)

SYMBOLS = np.array((-3-3j, -3-1j, -3+1j, -3+3j, -1-3j, -1-1j, -1+1j, -1+3j, 1-3j, 1-1j, 1+1j, 1+3j, 3-3j, 3-1j, 3+1j, 3+3j))
out = {}
cases = [("wtx", 16, 8, 0, 21), ("CPW", 22, 8, 10, 22), ("wrx", 10, 0, 10, 23)]
for k, (name, cp, ttx, trx, seed) in enumerate(cases):
    p = O.system_params(name, 256, cp, ttx, trx, S=16, bits=4)
    vt = O.perturbed_windows(p, seed=seed)[0]
    model = wOFDMSystem(name, 256, cp, ttx, trx, "/tmp")
    assert model.cs_len == p.cs
    np.random.seed(seed)
    opt, rc, cpd = model.estimate_obr(np.diagflat(vt), 200e-9)
    np.random.seed(seed)
    X = np.random.choice(SYMBOLS, size=(256 - 96, 256), replace=True)
    idx = np.array([int(np.argmin(np.abs(SYMBOLS - v))) for v in X.ravel()]).reshape(X.shape)
    out[f"c{k}_name"] = np.array(name); out[f"c{k}_cp"] = cp; out[f"c{k}_ttx"] = ttx; out[f"c{k}_trx"] = trx
    out[f"c{k}_win_tx"] = vt; out[f"c{k}_idx"] = idx.astype(np.int8)
    out[f"c{k}_X_opt"] = opt["X_est_opt"]; out[f"c{k}_X_rc"] = rc["X_est_rc"]; out[f"c{k}_X_cp"] = cpd["X_est_cp"]
    out[f"c{k}_S_opt"] = opt["S_opt"]; out[f"c{k}_S_rc"] = rc["S_rc"]; out[f"c{k}_S_cp"] = cpd["S_cp"]
    out[f"c{k}_obr"] = np.array([opt["obr_opt"], rc["obr_rc"], cpd["obr_cp"]])
out["n_cases"] = len(cases)
np.savez_compressed(os.path.join(HERE, "psd.npz"), **out)
print("wrote psd.npz", os.path.getsize(os.path.join(HERE, "psd.npz")))
