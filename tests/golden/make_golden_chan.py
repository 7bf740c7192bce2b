"""Golden vectors for the channel generator (SURVEY 8f-4), produced by executing the REFERENCE's
channel_model.gen_chan (python/channel_model/itur_channels.py:33-94) under np.random.seed; the phases it drew are
recovered by replaying the same seed (np.random.randn(1) per oscillator part, rayleigh_fading.py:95-98).

Run:  WOFDM_REFERENCE=<checkout of felipescoelho/w-ofdm-optimization> python -B tests/golden/make_golden_chan.py"""
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.environ["WOFDM_REFERENCE"], "python"))
import numpy as np  # noqa: E402
from channel_model.itur_channels import gen_chan, CHANNEL_ITUR  # noqa: E402

out = {}
fd = (100 / 3.6 / 299792458.0) * 2e9           # wofdm_optimization.py:63-76
fs = 1 / 200e-9
frame = 16 * 256 * 200e-9
cases = [("vehicularA", 21, 1, 11), ("vehicularA", 21, 7, 12), ("vehicularB", 33, 5, 13),
         ("outdoor-indoorA", 21, 3, 14), ("outdoor-indoorB", 16, 64, 15)]
for k, (std, L, frames, seed) in enumerate(cases):
    n_paths = len(CHANNEL_ITUR[std]["relative_delay"])
    np.random.seed(seed)
    taps = gen_chan(std, L, fd, fs, frame, frames)
    np.random.seed(seed)
    phases = np.array([np.random.randn(1)[0] for _ in range(n_paths * 21 * 2)]).reshape(n_paths, 21, 2)
    out[f"c{k}_std"] = np.array(std); out[f"c{k}_L"] = L; out[f"c{k}_frames"] = frames
    out[f"c{k}_phases"] = phases; out[f"c{k}_taps"] = taps
out["n_cases"] = len(cases); out["fd"] = fd; out["fs"] = fs; out["frame"] = frame
np.savez_compressed(os.path.join(HERE, "chan_gen.npz"), **out)
print("wrote chan_gen.npz", {k: v.shape for k, v in out.items() if k.endswith("taps")})
