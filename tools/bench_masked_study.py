"""The channel-mask study's calls for several configurations against the single calls they replace.

  * adaptive: wofdm_ber_run_masked_adaptive_multi (n_var = 1, 2, 8) against n_var single wofdm_ber_run_masked_adaptive
    calls, at bench.py's mask_chain shape (wtx N = 256, cp 16, tail_tx 8, guard 64, 250 channels x 30 SNR points,
    ensemble_max 16, MATLAB conventions).  With a target no point reaches both arms run the same frames (the comparable
    number: a real target stops a point of the multi call only when every configuration has reached it); wall time with
    host buffers, alternated, median of --rounds rounds; the unmasked rows are checked equal to the single calls' in the
    same run.  A real-target run is reported separately, with the frames each arm ran;
  * PSD: wofdm_psd_masked_multi (n_var = 1, 2, 8) against n_var single wofdm_psd_masked calls (wtx N = 256, S = 256, 4096
    frames, reference estimator), spectra checked against the single calls to 1e-12; with --parent-lib (a build of the
    parent commit's libwofdm.so), the single call against that build's, alternated in the same process;
  * pair v: the RC windows (v = 0) or RC perturbed by a seeded +-10 %; roll-offs {4, 6, 8, 10, 14, 20, 30, 40} in that order;
  * the card's name and power limit, read in the same run.
Writes one JSON record to --out."""
import argparse
import ctypes as C
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
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--nvars", default="1,2,8")
ap.add_argument("--target", type=int, default=20000, help="bit-error target of the real-target run")
ap.add_argument("--psd-frames", type=int, default=4096)
ap.add_argument("--parent-lib", help="libwofdm.so of the parent commit: its wofdm_psd_masked as the PSD baseline")
ap.add_argument("--out", required=True)
a = ap.parse_args()

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
ROLL_OFFS = [4, 6, 8, 10, 14, 20, 30, 40]
nvars = [int(x) for x in a.nvars.split(",")]
s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1, guard=64)
p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
rng = np.random.default_rng(0)                          # bench.py's mask_chain channels and SNR points
chan = (rng.standard_normal((21, 250)) + 1j * rng.standard_normal((21, 250))) * np.exp(-np.arange(21) / 4)[:, None]
snr = np.linspace(-20, 50, 30)
E = 16
wt, wr = [capi.rc_window_tx(s)], [capi.rc_window_rx(s)]
for v in range(1, 8):
    vt, vr, _, _ = O.perturbed_windows(p, seed=100 + v)
    wt.append(vt)
    wr.append(vr)
wt, wr = np.array(wt), np.array(wr)
h = W.Handle([0])


def stats(t):
    t = np.asarray(t) * 1e3
    return {"median": float(np.median(t)), "min": float(t.min()), "max": float(t.max())}


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, time.perf_counter() - t0


# ---- adaptive -----------------------------------------------------------------------------------------------------------
def ad_multi(nv, seed, target):
    return h.ber_run_masked_adaptive_multi(s, wt[:nv], wr[:nv], chan, snr, E, target_bit_errors=target, seed=seed,
                                           roll_offs=ROLL_OFFS[:nv])


def ad_singles(nv, seed, target):
    return [h.ber_run_masked_adaptive(s, wt[v], wr[v], chan, snr, E, target_bit_errors=target, seed=seed, variant=v,
                                      roll_off=ROLL_OFFS[v]) for v in range(nv)]


NEVER = 10 ** 15
adaptive = {}
for nv in nvars:                                   # warm-up
    ad_multi(nv, 1, NEVER), ad_singles(nv, 1, NEVER)
times = {}
equal = {nv: True for nv in nvars}
for rd in range(a.rounds):                         # alternated: multi, then singles, for every n_var
    for nv in nvars:
        m, dt = timed(lambda: ad_multi(nv, 2 + rd, NEVER))
        times.setdefault((nv, "multi"), []).append(dt)
        r, dt = timed(lambda: ad_singles(nv, 2 + rd, NEVER))
        times.setdefault((nv, "singles"), []).append(dt)
        # (unmasked pair v: noise stream v in both arms; the masked streams differ, n_var + v against v + 1)
        equal[nv] &= all(np.array_equal(m["bit_err"][1, v], r[v]["bit_err"][1]) for v in range(nv))
for nv in nvars:
    tm, ts = times[(nv, "multi")], times[(nv, "singles")]
    adaptive[str(nv)] = {"multi_ms": stats(tm), "singles_ms": stats(ts), "multi_over_singles": float(np.median(tm) / np.median(ts)),
                         "frames_per_chain_and_pair": int(250 * 30 * E), "unmasked_rows_equal_every_round": equal[nv],
                         "roll_offs": ROLL_OFFS[:nv]}
real = {}
for nv in nvars:                                   # one timed call of each arm with a real target
    m, tm = timed(lambda: ad_multi(nv, 7, a.target))
    r, ts = timed(lambda: ad_singles(nv, 7, a.target))
    real[str(nv)] = {"multi_ms": tm * 1e3, "singles_ms": ts * 1e3,
                     "multi_frames_per_chain_and_pair": int(m["ensemble_used"].sum() * 250),
                     "singles_frames_per_chain": [int(x["ensemble_used"].sum() * 250) for x in r],
                     "multi_rounds": m["rounds"], "singles_rounds": [x["rounds"] for x in r]}

# ---- PSD ----------------------------------------------------------------------------------------------------------------
sp = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=256, noise_norm=1, constellation=1, guard=64)
F = a.psd_frames


def psd_multi(nv):
    return h.psd_masked_multi(sp, wt[:nv], roll_offs=ROLL_OFFS[:nv], frames=F, seed=3)


def psd_singles(nv):
    return [h.psd_masked(sp, wt[v], roll_off=ROLL_OFFS[v], frames=F, seed=3) for v in range(nv)]


class ParentPsd:
    """wofdm_psd_masked of another build of the library, on a handle of its own"""
    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.wofdm_psd_masked.argtypes = capi.SIGNATURES["wofdm_psd_masked"][1]
        self.h = C.c_void_p()
        ids = (C.c_int * 1)(0)
        assert self.lib.wofdm_create_on(C.byref(self.h), ids, 1) == 0

    def __call__(self, v):
        om, ou = np.empty(8 * sp.N), np.empty(8 * sp.N)
        w = np.ascontiguousarray(wt[v])
        assert self.lib.wofdm_psd_masked(self.h, C.byref(sp), w.ctypes.data_as(capi._dp), ROLL_OFFS[v], 3, 0, F, 0,
                                         om.ctypes.data_as(capi._dp), ou.ctypes.data_as(capi._dp)) == 0
        return om, ou


psd = {}
for nv in nvars:
    mm, mu = psd_multi(nv)
    r = psd_singles(nv)
    dev = max(float(np.max(np.abs(x[v] - r[v][k]) / np.abs(r[v][k]))) for v in range(nv) for k, x in enumerate((mm, mu)))
    times = {"multi": [], "singles": []}
    for rd in range(a.rounds):
        times["multi"].append(timed(lambda: psd_multi(nv))[1])
        times["singles"].append(timed(lambda: psd_singles(nv))[1])
    psd[str(nv)] = {"multi_ms": stats(times["multi"]), "singles_ms": stats(times["singles"]),
                    "multi_over_singles": float(np.median(times["multi"]) / np.median(times["singles"])),
                    "max_relative_deviation_from_singles": dev, "roll_offs": ROLL_OFFS[:nv]}
parent = None
if a.parent_lib:
    old = ParentPsd(a.parent_lib)
    ref = old(0)
    new = h.psd_masked(sp, wt[0], roll_off=ROLL_OFFS[0], frames=F, seed=3)
    dev = max(float(np.max(np.abs(x - y) / np.abs(y))) for x, y in zip(new, ref))
    t_old, t_new = [], []
    for rd in range(max(a.rounds, 7)):
        t_old.append(timed(lambda: old(0))[1])
        t_new.append(timed(lambda: h.psd_masked(sp, wt[0], roll_off=ROLL_OFFS[0], frames=F, seed=3))[1])
    parent = {"this_ms": stats(t_new), "parent_ms": stats(t_old), "this_over_parent": float(np.median(t_new) / np.median(t_old)),
              "max_relative_deviation": dev}

rec = {"card": card,
       "adaptive_shape": "bench.py mask_chain: wtx N=256 cp=16 tail_tx=8 guard=64, S=16, 16-QAM, 250 channels x 30 SNR points, "
                         "ensemble_max 16, first_block 1, MATLAB conventions",
       "adaptive_unreachable_target": adaptive, "adaptive_real_target": {"target_bit_errors": a.target, "cases": real},
       "psd_shape": f"wtx N=256 cp=16 tail_tx=8 guard=64, S=256, 16-QAM, {F} frames, reference estimator, both halves",
       "psd": psd, "psd_single_against_parent": parent,
       "rounds": a.rounds, "wall": "host buffers in, host arrays out; median of alternated rounds"}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as fh:
    json.dump(rec, fh, indent=1)
print(json.dumps(rec, indent=1))
h.close()
