"""The K1 production kernels with SEVERAL frames per CTA (the reuse of shared memory from frame to frame without a closing
barrier is what a race checker should look at), small enough for `compute-sanitizer --tool racecheck`:
    compute-sanitizer --tool racecheck python tools/sanitize_k1.py [n256|multi|wtx|n1024]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import wofdm_b200 as W
from wofdm_b200 import capi

which = sys.argv[1] if len(sys.argv) > 1 else "n256"
rng = np.random.default_rng(0)
h = W.Handle([0])
chan = rng.standard_normal((21, 3)) + 1j * rng.standard_normal((21, 3))
snr = np.array([5.0, 25.0])
if which == "n512":
    s = W.params_from_name("CPW", 512, 32, 16, 20, bits=6, S=16, noise_norm=1, constellation=1)
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    r = h.ber_run(s, vt, vr, chan, snr, 80, seed=1)                      # 480 frames on 148 CTAs
elif which == "wtx":                                                     # the fixed-shape instance (ber_tconv2.cuh: HS)
    s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1)
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    plan = h.ber_plan(s, vt, vr, chan, snr)
    print("KERNEL", plan.kernel)
    plan.close()
    r = h.ber_run(s, vt, vr, chan, snr, 150, seed=1)                     # 900 frames on <= 296 CTAs
elif which in ("n256", "multi"):
    s = W.params_from_name("WOLA", 256, 16, 8, 10, bits=4, S=16, noise_norm=0, constellation=0)
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    if which == "n256":
        r = h.ber_run(s, vt, vr, chan, snr, 150, seed=1)                 # 900 frames on <= 296 CTAs
    else:
        r = h.ber_run_multi(s, [vt, vt * 0.9], [vr, vr], chan, snr, 150, seed=1)
else:
    s = W.params_from_name("WOLA", 1024, 64, 32, 40, bits=6, S=16, noise_norm=0, constellation=0)
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    r = h.ber_run(s, vt, vr, chan, snr, 40, seed=1)                      # 240 frames on 74 clusters
print(which, "SER", np.round(r["sym_err"] / r["sym_tot"], 4))
print("COUNTERS", which, np.asarray(r["bit_err"]).ravel().tolist(), np.asarray(r["sym_err"]).ravel().tolist())
