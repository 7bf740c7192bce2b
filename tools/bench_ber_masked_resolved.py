"""Cost of resolving the channel-mask chain's counters (wofdm_ber_run_masked_resolved) against the unresolved chain
(wofdm_ber_run_masked).

bench.py's mask_chain shape: main_channel_mask.m run_sim_mc, wtx-OFDM N = 256, cp 16, tail_tx 8, 16-QAM, 128 active
sub-carriers (guard 64), RC mask roll-off 10 bins, 250 channels x 30 SNR points x ensemble 16 = 120 000 frames, MATLAB
conventions.  The same job four ways in one process -- unresolved, by sub-carrier, by channel, by both -- warmed up, then
alternated for --reps rounds; each call's wall time ends in a device synchronise (the counters are read back).  The sum
identity is checked on every call.  A separate pass under torch.profiler (after the timed rounds, one call per mode) gives
the device time of the K1 kernels alone and of the whole call's kernels, so that kernel cost and per-call cost can be told
apart.  The card's name and power limit are read in the same run.  One JSON line on stdout (and in --out)."""
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


def workload():
    """bench.py's mask_chain inputs."""
    s = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1, guard=64)
    rng = np.random.default_rng(0)
    ch = (rng.standard_normal((21, 250)) + 1j * rng.standard_normal((21, 250))) * np.exp(-np.arange(21) / 4)[:, None]
    snr = np.linspace(-20, 50, 30)
    return s, W.capi.rc_window_tx(s), W.capi.rc_window_rx(s), ch, snr, 16


def profile_kernels(call):
    """Per mode: device time (ms) of the K1 launches (ber_tconv2_kernel / ber_frame_kernel) and of every kernel of one
    call, from a torch.profiler trace with CUDA activities; {} when torch or its CUDA profiler is not available."""
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
        k1 = every = 0.0
        for e in prof.events():             # (kernel records: device-side events, their own interval)
            if "CPU" in str(e.device_type) or "memcpy" in e.name.lower() or "memset" in e.name.lower():
                continue
            every += e.time_range.elapsed_us()
            if "ber_tconv2_kernel" in e.name or "ber_frame_kernel" in e.name:
                k1 += e.time_range.elapsed_us()
        out[mode] = (k1 / 1e3, every / 1e3)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=7, help="alternated rounds of the four calls")
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    a = ap.parse_args()
    info = card()
    s, vt, vr, ch, snr, ens = workload()
    with W.Handle([0]) as h:
        def call(mode):
            if MODES[mode] is None:
                return h.ber_run_masked(s, vt, vr, ch, snr, ens, seed=2, variant=1)
            b, c = MODES[mode]
            return h.ber_run_masked_resolved(s, vt, vr, ch, snr, ens, seed=2, variant=1, by_subcarrier=b, by_channel=c)

        def check(mode, r):
            if mode != "unresolved":
                for key in ("bit_err", "sym_err"):
                    assert np.array_equal(r[key].sum(axis=(1, 2)), ref[key]), (mode, key)

        os.environ["WOFDM_DEBUG"] = "1"                  # (the kernel names go to stderr once)
        ref = call("unresolved")
        for mode in MODES:                               # warm-up: modules, arenas, every shape of the timed window
            check(mode, call(mode))
        del os.environ["WOFDM_DEBUG"]
        times = {m: [] for m in MODES}
        for _ in range(a.reps):
            for mode in MODES:                           # alternated: drifts of the shared host hit every mode alike
                t0 = time.perf_counter()
                r = call(mode)
                times[mode].append(time.perf_counter() - t0)
                check(mode, r)
        dev_ms = profile_kernels(call)
    frames = len(snr) * ch.shape[1] * ens
    syms = frames * s.S
    base = float(np.median(times["unresolved"]))
    modes = {}
    for mode, t in times.items():
        med = float(np.median(t))
        modes[mode] = dict(median_ms=round(med * 1e3, 3), min_ms=round(float(np.min(t)) * 1e3, 3),
                           max_ms=round(float(np.max(t)) * 1e3, 3), ofdm_symbols_per_s=float(f"{syms / med:.4g}"),
                           call_cost_vs_unresolved=round(med / base - 1.0, 4))
        if dev_ms:
            k1, every = dev_ms[mode]
            modes[mode].update(k1_kernel_ms=round(k1, 3), all_kernels_ms=round(every, 3),
                               k1_kernel_cost_vs_unresolved=round(k1 / dev_ms["unresolved"][0] - 1.0, 4),
                               all_kernels_cost_vs_unresolved=round(every / dev_ms["unresolved"][1] - 1.0, 4))
    rec = dict(metric="channel-mask chain, resolved counters: call wall time and K1 device time against wofdm_ber_run_masked",
               card=info, workload="bench.py mask_chain: wtx N=256 cp=16 tail_tx=8 16-QAM, guard 64, roll-off 10, "
                                   f"{ch.shape[1]} channels x {len(snr)} SNR points x ensemble {ens} = {frames} frames",
               timing="wall time of each C-ABI call (host setup, mask product, K1, device synchronise, counter read-back); "
                      f"median of {a.reps} alternated rounds after one warm-up call per mode; device times from a separate "
                      "torch.profiler pass, one call per mode",
               errors=int(ref["sym_err"].sum()), modes=modes)
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
