"""Small production + verify runs of every tuned K1 policy plus one TF32 interference call: the workload to put under
`compute-sanitizer --tool memcheck|racecheck|synccheck python tools/sanitize_small.py` where that tool is available
(it is closed on the round-1 GPU pool; tests/test_ber_frame_invariance.py is the stand-in there)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import wofdm_b200 as W
from wofdm_b200 import capi

rng = np.random.default_rng(0)
h = W.Handle([0])
cases = [("wtx", 256, 16, 8, 0, 4), ("CPW", 256, 16, 8, 10, 4), ("WOLA", 1024, 64, 32, 40, 6), ("CPW", 1024, 64, 32, 40, 6), ("WOLA", 64, 8, 2, 2, 2)]
for name, N, cp, ttx, trx, bits in cases:
    for nn, conv in ((0, 0), (1, 1)):
        s = W.params_from_name(name, N, cp, ttx, trx, bits=bits, S=16, noise_norm=nn, constellation=conv)
        vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
        chan = rng.standard_normal((21, 3)) + 1j * rng.standard_normal((21, 3))
        r = h.ber_run(s, vt, vr, chan, np.array([5.0, 25.0]), 3, seed=1)
        F = 2
        sym = rng.integers(0, 1 << bits, size=(F, 16, N))
        nl = s.noise_len(21)
        nz = rng.standard_normal((F, nl)) + 1j * rng.standard_normal((F, nl))
        eq, dec, be, se = h.ber_verify(s, vt, vr, chan[:, :F], np.array([10.0, 20.0]), sym, nz)
        eq2, dec2, be2, se2 = h.ber_verify(s, vt, vr, chan[:, :F], np.array([10.0, 20.0]), sym, nz, direct=True)
        print(name, N, nn, "ser", np.round(r["sym_err"] / r["sym_tot"], 3), "verify sym_err", se, se2)
P = h.interf_power(W.params_from_name("WOLA", 256, 16, 8, 10, precision=1), capi.rc_window_tx(W.params_from_name("WOLA", 256, 16, 8, 10)),
                   capi.rc_window_rx(W.params_from_name("WOLA", 256, 16, 8, 10)), rng.standard_normal((21, 4)) + 0j, mode=1)
print("interf tf32", P.sum())
