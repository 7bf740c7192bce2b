"""Throughput of wofdm_psd_masked at bench.py's mask_chain shape with long records (wtx, N = 256, cp 16, tail 8, guard 64,
roll-off 10, S = 256 symbols per frame, MATLAB conventions), both estimators, 4096 frames (1.05e6 OFDM symbols) per call.

  * wall time of the call with host buffers (both spectra), median of alternated rounds, at the library's product batch
    (131072 symbols);
  * device time per kernel (symbol kernel, product, psd_masked_kernel) from a separate torch.profiler pass, and the PSD
    kernel's rate over the bytes of Y it must read (every filtered symbol's n_tx complex fp32 samples once, for each of
    the two spectra);
  * the card's name and power limit, read in the same run.
Writes one JSON record to --out."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import wofdm_b200 as W
from wofdm_b200 import capi

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=4096)
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--out", required=True)
a = ap.parse_args()

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=256, noise_norm=1, constellation=1, guard=64)
vt = capi.rc_window_tx(s)
F = a.frames
h = W.Handle([0])
times = {}
for est in ("reference", "hann"):                # warm-up of both estimators
    h.psd_masked(s, vt, frames=F, seed=1, estimator=est)
for r in range(a.rounds):                        # alternated estimators
    for est in ("reference", "hann"):
        t0 = time.perf_counter()
        xm, xu = h.psd_masked(s, vt, frames=F, seed=2 + r, estimator=est)
        times.setdefault(est, []).append(time.perf_counter() - t0)
wall = {k: {"median_ms": float(np.median(v) * 1e3), "min_ms": float(np.min(v) * 1e3), "max_ms": float(np.max(v) * 1e3),
            "ofdm_symbols_per_s": float(F * s.S / np.median(v))} for k, v in times.items()}

# levels of the last call (Hann) relative to the in-band mean
gb, P = 8 * s.guard, 8 * s.N
deep = np.r_[0:gb - 256, P - gb + 256:P]
levels = {}
for name, x in (("masked", xm), ("unmasked", xu)):
    inb = x[gb + 16:P - gb - 16].mean()
    levels[name] = {"obr_db": float(10 * np.log10(np.r_[x[:gb], x[-gb:]].mean() / inb)),
                    "deep_oob_db": float(10 * np.log10(x[deep].mean() / inb))}

# device time per kernel: a separate profiled pass
import torch
from torch.profiler import ProfilerActivity, profile

kern = {}
for est in ("reference", "hann"):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.psd_masked(s, vt, frames=F, seed=3, estimator=est)
    torch.cuda.synchronize()
    k = kern.setdefault(est, {})
    for e in prof.key_averages():
        for tag in ("mask_sym_kernel", "mask_gemm_f16", "mask_matrix_kernel", "mask_split_kernel", "psd_masked_kernel"):
            if tag in e.key:
                d = k.setdefault(tag, {"device_ms": 0.0, "launches": 0})
                d["device_ms"] += e.device_time_total / 1e3
                d["launches"] += e.count
y_bytes = 2 * F * s.S * s.n_tx * 8                                 # both spectra: every symbol's n_tx complex fp32 once
for est, k in kern.items():
    psd_ms = k["psd_masked_kernel"]["device_ms"]
    k["psd_kernel_y_read_GBps"] = y_bytes / (psd_ms * 1e-3) / 1e9
    k["psd_over_product_time"] = psd_ms / k["mask_gemm_f16"]["device_ms"]
rec = {"card": card, "shape": "wtx N=256 cp=16 tail_tx=8 guard=64 roll-off 10, S=256, 16-QAM (MATLAB conventions)",
       "frames_per_call": F, "ofdm_symbols_per_call": F * s.S, "default_batch_cols": 131072,
       "wall_host_buffers": wall, "rounds": a.rounds,
       "device_time_per_call_default_batch": kern, "psd_kernel_y_bytes_per_call": y_bytes,
       "levels_hann_last_call": levels}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as fh:
    json.dump(rec, fh, indent=1)
print(json.dumps(rec, indent=1))
h.close()
