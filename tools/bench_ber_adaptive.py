"""Cost and savings of the stopping rule (wofdm_ber_run_adaptive) against the fixed-ensemble chain (wofdm_ber_run_multi).

bench.py's configs[1] shapes: wtx-OFDM N = 256, 16-QAM, 250 channels, 30 SNR points from -20 to 50 dB, two window pairs per
frame (the optimised stand-in and RC), ensemble_max 27 and 432.  Per ensemble_max, in one process:
  fixed        wofdm_ber_run_multi(ensemble = ensemble_max)
  unreachable  adaptive with a target no point reaches, first_block 1 (the most rounds) and first_block = ensemble_max
               (one round: the twin kernel's own cost); both must equal the fixed run's counters
  sym100, sym1000, bit1000, sym1000000   adaptive with those targets, first_block 1 (one ensemble index of this
               workload already counts >= 25 000 symbol errors at every point; the last target takes several rounds)
Each mode is warmed up, then the modes are alternated for --reps rounds; each call's wall time ends in a device synchronise
(the counters are read back).  Reports wall times, the cost against the fixed run, rounds, frames per point and in total,
and reads the card's name and power limit in the same run.  One JSON line on stdout (and in --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True
import wofdm_b200 as W  # noqa: E402
from bench import CFG, windows_for, workload_inputs  # noqa: E402
from bench_ber_resolved import card  # noqa: E402

UNREACHABLE = 10 ** 18


def run_case(h, ensemble_max, reps):
    cfg = CFG
    s = W.capi.params_from_name(cfg["system"], cfg["N"], cfg["cp"], cfg["tail_tx"], cfg["tail_rx"], bits=cfg["bits"],
                                S=cfg["S"], noise_norm=cfg["noise_norm"], constellation=cfg["constellation"])
    chan, snr = workload_inputs(cfg, h)
    wt, wr = windows_for(cfg, W.capi, s)
    wins_tx, wins_rx = [wt, W.capi.rc_window_tx(s)], [wr, W.capi.rc_window_rx(s)]
    C = chan.shape[1]
    modes = {
        "fixed": lambda: h.ber_run_multi(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3),
        "unreachable_first_block_1": lambda: h.ber_run_adaptive(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3,
                                                                target_symbol_errors=UNREACHABLE, first_block=1),
        "unreachable_one_round": lambda: h.ber_run_adaptive(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3,
                                                            target_symbol_errors=UNREACHABLE, first_block=ensemble_max),
        "sym100": lambda: h.ber_run_adaptive(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3, target_symbol_errors=100),
        "sym1000": lambda: h.ber_run_adaptive(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3, target_symbol_errors=1000),
        "bit1000": lambda: h.ber_run_adaptive(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3, target_bit_errors=1000),
        "sym1000000": lambda: h.ber_run_adaptive(s, wins_tx, wins_rx, chan, snr, ensemble_max, seed=3,
                                                 target_symbol_errors=10 ** 6),
    }
    res = {m: f() for m, f in modes.items()}                      # warm-up, and the results the record describes
    ref = res["fixed"]
    for m in ("unreachable_first_block_1", "unreachable_one_round"):
        for key in ("bit_err", "sym_err", "sym_tot"):
            assert np.array_equal(res[m][key], ref[key]), (m, key)
    times = {m: [] for m in modes}
    for _ in range(reps):
        for m, f in modes.items():                                # alternated: drifts of the shared host hit every mode alike
            t0 = time.perf_counter()
            f()
            times[m].append(time.perf_counter() - t0)
    base = float(np.median(times["fixed"]))
    out = dict(ensemble_max=ensemble_max, channels=C, n_snr=len(snr), pairs=2,
               fixed_frames=len(snr) * C * ensemble_max, modes={})
    for m, t in times.items():
        med = float(np.median(t))
        rec = dict(median_s=round(med, 5), min_s=round(float(np.min(t)), 5), max_s=round(float(np.max(t)), 5),
                   time_vs_fixed=round(med / base, 4))
        if m != "fixed":
            used = res[m]["ensemble_used"]
            rec.update(rounds=int(res[m]["rounds"]), frames_per_point=[int(u) * C for u in used],
                       total_frames=int(used.sum()) * C, frames_vs_fixed=round(float(used.sum()) / (len(snr) * ensemble_max), 4),
                       min_errors_per_point=[int(x) for x in (res[m]["bit_err"] if m == "bit1000" else res[m]["sym_err"]).min(axis=0)])
        out["modes"][m] = rec
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5, help="alternated rounds of the calls")
    ap.add_argument("--ensembles", default="27,432", help="ensemble_max values")
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    a = ap.parse_args()
    info = card()
    with W.Handle([0]) as h:
        cases = [run_case(h, int(e), a.reps) for e in a.ensembles.split(",")]
    rec = dict(metric="stopping rule of the BER chain: wall time and frames against wofdm_ber_run_multi", card=info,
               workload="configs[1] shapes (wtx N=256, 16-QAM, 250 channels, 30 SNR points -20..50 dB), 2 window pairs",
               timing="wall time of each C-ABI call (host setup, launches, device synchronise, counter read-back); median of "
                      f"{a.reps} alternated rounds after one warm-up call per mode", cases=cases)
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
