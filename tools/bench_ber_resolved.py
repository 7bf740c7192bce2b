"""Cost of resolving the BER counters (wofdm_ber_run_resolved) against the unresolved chain (wofdm_ber_run_multi).

bench.py's step shape: configs[1] (wtx-OFDM N = 256, 16-QAM, 250 channels, 30 SNR points, ensemble 27 x 16), two window
pairs per frame (the optimised stand-in and RC).  The same job four ways in one process -- unresolved, by sub-carrier,
by channel, by both -- warmed up, then alternated for --reps rounds; each call's wall time ends in a device synchronise
(the counters are read back).  Also one configs[4] case (WOLA N = 1024, 64-QAM; --c4-channels of its 10 000 channels).
Reports OFDM symbols/s (frames x S x pairs per second) per mode and the cost relative to the unresolved call, checks the
sum identity on every call, and reads the card's name and power limit in the same run.  A separate pass under
torch.profiler (after the timed rounds, one call per mode) gives the device time of the K1 kernels alone, so that kernel
cost and per-call cost can be told apart.  One JSON line on stdout (and in
--out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True
import wofdm_b200 as W  # noqa: E402
from bench import CFG, CFG4, windows_for, workload_inputs  # noqa: E402

MODES = {"unresolved": None, "subcarrier": (True, False), "channel": (False, True), "both": (True, True)}


def card():
    dev = (os.environ.get("CUDA_VISIBLE_DEVICES") or "0").split(",")[0]
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        out = subprocess.run(q + (["-i", dev] if dev.isdigit() else []), capture_output=True, text=True, check=True).stdout
        name, power, clock = (x.strip() for x in out.strip().splitlines()[0].split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except (OSError, subprocess.CalledProcessError, ValueError):
        return dict(name="unknown", power_limit="unknown", max_sm_clock="unknown")


def run_case(h, cfg, ensemble, C, reps):
    s = W.capi.params_from_name(cfg["system"], cfg["N"], cfg["cp"], cfg["tail_tx"], cfg["tail_rx"], bits=cfg["bits"],
                                S=cfg["S"], noise_norm=cfg["noise_norm"], constellation=cfg["constellation"])
    chan, snr = workload_inputs(dict(cfg, C=C), h)
    wt, wr = windows_for(cfg, W.capi, s)
    wins_tx, wins_rx = [wt, W.capi.rc_window_tx(s)], [wr, W.capi.rc_window_rx(s)]
    kernel = h.ber_plan_multi(s, wins_tx, wins_rx, chan, snr).kernel

    def call(mode):
        if MODES[mode] is None:
            return h.ber_run_multi(s, wins_tx, wins_rx, chan, snr, ensemble, seed=3)
        b, c = MODES[mode]
        return h.ber_run_resolved(s, wins_tx, wins_rx, chan, snr, ensemble, seed=3, by_subcarrier=b, by_channel=c)

    ref = call("unresolved")
    for mode in MODES:                                   # warm-up: modules, arenas, every shape of the timed window
        r = call(mode)
        if mode != "unresolved":
            assert np.array_equal(r["sym_err"].sum(axis=(2, 3)), ref["sym_err"]), mode
            assert np.array_equal(r["bit_err"].sum(axis=(2, 3)), ref["bit_err"]), mode
    times = {m: [] for m in MODES}
    for _ in range(reps):
        for mode in MODES:                               # alternated: drifts of the shared host hit every mode alike
            t0 = time.perf_counter()
            r = call(mode)
            times[mode].append(time.perf_counter() - t0)
            if mode != "unresolved":
                assert np.array_equal(r["sym_err"].sum(axis=(2, 3)), ref["sym_err"]), mode
    kernel_ms = profile_kernels(call)
    frames = len(snr) * C * ensemble
    syms = frames * cfg["S"] * 2
    base = float(np.median(times["unresolved"]))
    out = dict(system=cfg["system"], N=cfg["N"], bits=cfg["bits"], S=cfg["S"], L=cfg["L"], channels=C, n_snr=len(snr),
               ensemble=ensemble, pairs=2, frames=frames, ofdm_symbols_per_call=syms, production_kernel=kernel,
               errors=int(ref["sym_err"].sum()), modes={})
    for mode, t in times.items():
        med = float(np.median(t))
        out["modes"][mode] = dict(median_s=round(med, 5), min_s=round(float(np.min(t)), 5), max_s=round(float(np.max(t)), 5),
                                  ofdm_symbols_per_s=float(f"{syms / med:.4g}"), cost_vs_unresolved=round(med / base - 1.0, 4))
        if kernel_ms:
            out["modes"][mode].update(k1_kernel_ms=round(kernel_ms[mode], 3),
                                      k1_kernel_cost_vs_unresolved=round(kernel_ms[mode] / kernel_ms["unresolved"] - 1.0, 4))
    return out


def profile_kernels(call):
    """Device time (ms) of the K1 kernel launches (ber_tconv2_kernel / ber_frame_kernel) of one call per mode, from a
    torch.profiler trace with CUDA activities; {} when torch or its CUDA profiler is not available."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
    except ImportError:
        return {}
    if not torch.cuda.is_available():
        return {}
    out = {}
    for mode in MODES:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(mode)
        t = 0.0
        for e in prof.events():             # (kernel records: device-side events, their own interval)
            if ("ber_tconv2_kernel" in e.name or "ber_frame_kernel" in e.name) and "CPU" not in str(e.device_type):
                t += e.time_range.elapsed_us()
        out[mode] = t / 1e3
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5, help="alternated rounds of the four calls")
    ap.add_argument("--c4-channels", type=int, default=1000, help="channels of the configs[4] case (BASELINE: 10 000)")
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    a = ap.parse_args()
    info = card()
    with W.Handle([0]) as h:
        c1 = run_case(h, CFG, CFG["ensemble"] * 16, CFG["C"], a.reps)
        c4 = run_case(h, CFG4, CFG4["ensemble"], a.c4_channels, a.reps)
    rec = dict(metric="resolved BER counters: OFDM symbols/s and cost against wofdm_ber_run_multi", card=info,
               timing="wall time of each C-ABI call (host setup, launch, device synchronise, counter read-back); median of "
                      f"{a.reps} alternated rounds after one warm-up call per mode", configs1=c1, configs4=c4)
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
