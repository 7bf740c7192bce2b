"""wofdm_ber_run_masked_multi against the single calls it replaces, at bench.py's mask_chain shape (wtx N = 256, cp 16, tail_tx
8, guard 64, 250 channels x 30 SNR points x ensemble 16 = 120 000 frames, MATLAB conventions).

  * cases n_var = 1, 2 and 8: pair 0 = the RC windows, pair v > 0 = RC perturbed by a seeded +-10 %; roll-offs
    {4, 6, 8, 10, 14, 20, 30, 40} in that order;
  * wall time with host buffers of ONE multi call against the n_var single ber_run_masked calls that give the same counters
    (pair v: its windows, roll-off and variant + v), alternated, median of --rounds rounds; the counters are checked equal
    in the same run;
  * device time per kernel (mask_sym_kernel, mask_gemm_f16, the K1 kernel, the stream assembly) and launches per call,
    from a separate torch.profiler pass of each arm;
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
from oracle import wofdm_oracle as O

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--nvars", default="1,2,8")
ap.add_argument("--out", required=True)
a = ap.parse_args()

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
ROLL_OFFS = [4, 6, 8, 10, 14, 20, 30, 40]
s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1, guard=64)
p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
rng = np.random.default_rng(0)                          # bench.py's mask_chain channels and SNR points
chan = (rng.standard_normal((21, 250)) + 1j * rng.standard_normal((21, 250))) * np.exp(-np.arange(21) / 4)[:, None]
snr = np.linspace(-20, 50, 30)
ens = 16
wt, wr = [capi.rc_window_tx(s)], [capi.rc_window_rx(s)]
for v in range(1, 8):
    vt, vr, _, _ = O.perturbed_windows(p, seed=100 + v)
    wt.append(vt)
    wr.append(vr)
wt, wr = np.array(wt), np.array(wr)
h = W.Handle([0])


def multi(nv, seed):
    return h.ber_run_masked_multi(s, wt[:nv], wr[:nv], chan, snr, ens, seed=seed, variant=1, roll_offs=ROLL_OFFS[:nv])


def singles(nv, seed):
    rs = [h.ber_run_masked(s, wt[v], wr[v], chan, snr, ens, seed=seed, variant=1 + v, roll_off=ROLL_OFFS[v]) for v in range(nv)]
    return {"bit_err": np.array([r["bit_err"] for r in rs]), "sym_err": np.array([r["sym_err"] for r in rs])}


nvars = [int(x) for x in a.nvars.split(",")]
for nv in nvars:                                   # warm-up, and the counters of both arms compared
    m, r = multi(nv, 1), singles(nv, 1)
    assert np.array_equal(m["bit_err"], r["bit_err"]) and np.array_equal(m["sym_err"], r["sym_err"]), nv
times = {}
equal = {nv: True for nv in nvars}
for rd in range(a.rounds):                         # alternated: multi, then singles, for every n_var
    for nv in nvars:
        t0 = time.perf_counter()
        m = multi(nv, 2 + rd)
        times.setdefault((nv, "multi"), []).append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        r = singles(nv, 2 + rd)
        times.setdefault((nv, "singles"), []).append(time.perf_counter() - t0)
        equal[nv] &= bool(np.array_equal(m["bit_err"], r["bit_err"]) and np.array_equal(m["sym_err"], r["sym_err"]))

frames = 250 * 30 * ens
cases = {}
for nv in nvars:
    tm, ts = np.array(times[(nv, "multi")]), np.array(times[(nv, "singles")])
    cases[str(nv)] = {"multi_ms": {"median": float(np.median(tm) * 1e3), "min": float(tm.min() * 1e3), "max": float(tm.max() * 1e3)},
                      "singles_ms": {"median": float(np.median(ts) * 1e3), "min": float(ts.min() * 1e3), "max": float(ts.max() * 1e3)},
                      "multi_over_singles": float(np.median(tm) / np.median(ts)),
                      "counters_equal_every_round": equal[nv],
                      "roll_offs": ROLL_OFFS[:nv]}

# device time per kernel: a separate profiled pass of each arm
import torch
from torch.profiler import ProfilerActivity, profile

TAGS = {"mask_sym_kernel": "mask_sym_kernel", "mask_gemm_f16": "mask_gemm_f16", "mask_assemble_kernel": "mask_assemble_kernel",
        "K1": ("ber_tconv2_kernel", "ber_kernel", "ber_staged"), "mask_setup": ("mask_response_kernel", "mask_matrix_kernel", "mask_split_kernel")}
for nv in nvars:
    for arm, fn in (("multi", multi), ("singles", singles)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn(nv, 9)
        torch.cuda.synchronize()
        k = {}
        for e in prof.key_averages():
            for tag, pat in TAGS.items():
                if any(x in e.key for x in ((pat,) if isinstance(pat, str) else pat)):
                    d = k.setdefault(tag, {"device_ms": 0.0, "launches": 0})
                    d["device_ms"] += e.device_time_total / 1e3
                    d["launches"] += e.count
                    if tag == "K1":
                        d["kernel"] = e.key
        k["sum_device_ms"] = sum(d["device_ms"] for d in k.values())
        cases[str(nv)]["device_" + arm] = k

rec = {"card": card,
       "shape": "bench.py mask_chain: wtx N=256 cp=16 tail_tx=8 guard=64, S=16, 16-QAM, 250 channels x 30 SNR points x ensemble 16, "
                "MATLAB conventions",
       "frames_per_call": frames, "rounds": a.rounds, "wall": "host buffers in, int64 counters out; median of alternated rounds",
       "cases": cases}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as fh:
    json.dump(rec, fh, indent=1)
print(json.dumps(rec, indent=1))
h.close()
