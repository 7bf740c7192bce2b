"""Cost of the channel-mask chain's stopping rule (wofdm_ber_run_masked_adaptive) against the two fixed calls run_sim_mc
makes (wofdm_ber_run_masked with variant 1, wofdm_ber_run with variant 0).

bench.py's mask_chain shape: main_channel_mask.m run_sim_mc, wtx-OFDM N = 256, cp 16, tail_tx 8, 16-QAM, 128 active
sub-carriers (guard 64), RC mask roll-off 10 bins, 250 channels x 30 SNR points, ensemble (ensemble_max) 16 = 120 000
frames per chain, MATLAB conventions.  In one process, warmed up, then alternated for --reps rounds: the two fixed calls
(timed together), an unreachable target with first_block 1 (five rounds of 1, 2, 4, 8, 1 indices) and 16 (one round), and
targets of 100, 1000 and 10^6 bit errors.  Each call's wall time ends in a device synchronise (the counters are read
back).  An unreachable target must return the fixed calls' counters bit for bit; that is checked on every call.  A separate
pass under torch.profiler (after the timed rounds, one call per mode) gives the device time of the K1 kernels and of all
kernels, so that the stopping rule's cost can be split into kernel time and host time.  The card's name and power limit are
read in the same run.  One JSON line on stdout (and in --out)."""
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


TARGET = 10 ** 18
MODES = {"fixed": None, "unreachable_fb1": (TARGET, 1), "unreachable_fb16": (TARGET, 16), "target_100": (100, 1),
         "target_1000": (1000, 1), "target_1e6": (10 ** 6, 1)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=7, help="alternated rounds of the calls")
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    a = ap.parse_args()
    info = card()
    s, vt, vr, ch, snr, ens = workload()
    with W.Handle([0]) as h:
        def call(mode):
            if MODES[mode] is None:
                m = h.ber_run_masked(s, vt, vr, ch, snr, ens, seed=2, variant=1)
                u = h.ber_run(s, vt, vr, ch, snr, ens, seed=2, variant=0)
                return dict(bit_err=np.stack([m["bit_err"], u["bit_err"]]), sym_err=np.stack([m["sym_err"], u["sym_err"]]),
                            ensemble_used=np.full(len(snr), ens), rounds=1)
            target, fb = MODES[mode]
            return h.ber_run_masked_adaptive(s, vt, vr, ch, snr, ens, target_bit_errors=target, first_block=fb, seed=2, variant=0)

        def check(mode, r):
            if mode.startswith("unreachable"):
                for key in ("bit_err", "sym_err"):
                    assert np.array_equal(r[key], ref[key]), (mode, key)

        ref = call("fixed")
        last = {}
        for mode in MODES:                               # warm-up: modules, arenas, every shape of the timed window
            check(mode, call(mode))
        times = {m: [] for m in MODES}
        for _ in range(a.reps):
            for mode in MODES:                           # alternated: drifts of the shared host hit every mode alike
                t0 = time.perf_counter()
                r = call(mode)
                times[mode].append(time.perf_counter() - t0)
                check(mode, r)
                last[mode] = r
        dev_ms = profile_kernels(call)
    C = ch.shape[1]
    base = float(np.median(times["fixed"]))
    modes = {}
    for mode, t in times.items():
        med = float(np.median(t))
        used = last[mode]["ensemble_used"]
        modes[mode] = dict(median_ms=round(med * 1e3, 3), min_ms=round(float(np.min(t)) * 1e3, 3),
                           max_ms=round(float(np.max(t)) * 1e3, 3), cost_vs_fixed=round(med / base - 1.0, 4),
                           rounds=int(last[mode]["rounds"]), frames_per_point_min=int(used.min()) * C,
                           frames_per_point_max=int(used.max()) * C, frames_total=int(used.sum()) * C,
                           fewest_bit_errors=int(last[mode]["bit_err"].min()))
        if dev_ms:
            k1, every = dev_ms[mode]
            modes[mode].update(k1_kernel_ms=round(k1, 3), all_kernels_ms=round(every, 3),
                               host_and_gaps_ms=round(med * 1e3 - every, 3),
                               k1_kernel_cost_vs_fixed=round(k1 / dev_ms["fixed"][0] - 1.0, 4),
                               all_kernels_cost_vs_fixed=round(every / dev_ms["fixed"][1] - 1.0, 4))
    rec = dict(metric="channel-mask chain, stopping rule: call wall time against the two fixed calls of run_sim_mc",
               card=info, workload="bench.py mask_chain: wtx N=256 cp=16 tail_tx=8 16-QAM, guard 64, roll-off 10, "
                                   f"{C} channels x {len(snr)} SNR points, ensemble_max {ens} "
                                   f"({len(snr) * C * ens} frames per chain)",
               timing="wall time of the C-ABI calls (host setup, mask product, K1 of both chains, device synchronise, counter "
                      f"read-back; 'fixed' = ber_run_masked + ber_run); median of {a.reps} alternated rounds after one "
                      "warm-up call per mode; device times from a separate torch.profiler pass, one call per mode; "
                      "host_and_gaps_ms = median wall time - device time of all kernels",
               modes=modes)
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
