"""Timing of the K1 kernel a plan picks, per case, on one GPU (development aid, not the bench).
usage: k1_ab.py [N] [ens]   -- env WOFDM_* select variants inside the library (a third argument, the kernel generations
of earlier versions of this script, is ignored)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import wofdm_b200 as W
from wofdm_b200 import capi

N = int(sys.argv[1]) if len(sys.argv) > 1 else 256
ens = int(sys.argv[2]) if len(sys.argv) > 2 else 27
scale = N // 256
h = W.Handle([0])
rng = np.random.default_rng(0)
C = 250
LT = int(os.environ.get("K1AB_L", "21"))       # channel taps
chan = (rng.standard_normal((LT, C)) + 1j * rng.standard_normal((LT, C))) * np.exp(-np.arange(LT) / 4)[:, None]
snr = np.linspace(-20, 50, 30)
stream = torch.cuda.Stream()
torch.cuda.set_stream(stream)
st = stream.cuda_stream
cases = [("wtx", 16, 0, 0), ("wtx", 16, 1, 1), ("WOLA", 16, 0, 0), ("CPW", 16, 0, 0), ("CP", 16, 0, 0), ("CPwtx", 10, 0, 0), ("wrx", 22, 0, 0)]
if N != 256:
    cases = [("WOLA", 16 * scale, 0, 0), ("CPW", 16 * scale, 0, 0), ("WOLA", 16 * scale, 1, 1)]
if os.environ.get("K1AB_CASES"):
    cases = [cases[int(i)] for i in os.environ["K1AB_CASES"].split(",")]
for name, cp, nn, conv in cases:
    ttx, trx = 8 * scale, 10 * scale
    if name in ("CP", "wrx", "CPwrx"): ttx = 0
    if name in ("CP", "wtx", "CPwtx"): trx = 0
    s = W.params_from_name(name, N, cp * (1 if N == 256 else 1), ttx, trx, bits=4 if N == 256 else 6, S=16, noise_norm=nn, constellation=conv)
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    plan = h.ber_plan(s, vt, vr, chan, snr)
    for _ in range(3):
        plan.launch(ens, seed=1, stream=st)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    K = 6
    e0.record()
    for k in range(K):
        plan.launch(ens, seed=2 + k, stream=st)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    syms = 30 * C * ens * 16
    be, se = plan.read()
    bt, stot = plan.totals(ens)
    ser = (se / stot)[[0, 15, 29]]
    print(f"{name:6s} cp={cp:3d} nn={nn} conv={conv} {plan.kernel:34s} {ms:8.3f} ms {syms / ms * 1e3:.4g} sym/s  SER {np.round(ser, 5)}", flush=True)
    plan.close()
h.close()
