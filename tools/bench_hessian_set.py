"""Window Hessian of a 250-channel set (wofdm_window_hessian_set) against 250 single-channel calls, WOLA at N = 256
(cp 16, tails 8 / 10: 54 variables), 21 taps.  One run, one JSON line on stdout (and in --out):
  set:     device time of one call (CUDA events from the first upload to the end of the download), the host time of the
           channel-set factorisation (reported separately, not part of the device time), passes, wall time of the call;
  single:  the sum over 250 wofdm_window_hessian calls of their device times, and their wall time;
  mean_ir: one call on the mean impulse response (what the reference optimises against).
Two sets: VehA channels (oracle.synth_channels: six paths sinc-interpolated onto 21 taps, covariance of rank 6) and a
full-rank set (independent taps, exponential profile: rank 21 = L, the most passes a set can take).  The set result is
checked against the mean of the 250 single-channel Hessians of the same run.  The card's name and power limit are read
in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import wofdm_b200 as W  # noqa: E402
from oracle import wofdm_oracle as O  # noqa: E402


def card():
    dev = (os.environ.get("CUDA_VISIBLE_DEVICES") or "0").split(",")[0]
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        out = subprocess.run(q + (["-i", dev] if dev.isdigit() else []), capture_output=True, text=True, check=True).stdout
        name, power, clock = (x.strip() for x in out.strip().splitlines()[0].split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except (OSError, subprocess.CalledProcessError, ValueError):
        return dict(name="unknown", power_limit="unknown", max_sm_clock="unknown")


def measure(h, s, chans, reps):
    C = chans.shape[1]
    h.window_hessian_set(s, chans)                                   # warm-up (arena, modules)
    dev, fac, wall = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        H = h.window_hessian_set(s, chans)
        wall.append((time.perf_counter() - t0) * 1e3)
        t = h.window_hessian_last_timing()
        dev.append(t["device_ms"]); fac.append(t["factor_ms"])
    passes = t["passes"]
    h.window_hessian(s, chans[:, 0])
    sdev, acc = 0.0, np.zeros_like(H)
    t0 = time.perf_counter()
    for c in range(C):
        acc += h.window_hessian(s, chans[:, c])
        sdev += h.window_hessian_last_timing()["device_ms"]
    swall = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    h.window_hessian(s, chans.mean(axis=1))
    mwall = (time.perf_counter() - t0) * 1e3
    mdev = h.window_hessian_last_timing()["device_ms"]
    ref = acc / C
    return dict(C=C, passes=passes,
                set_device_ms=float(np.median(dev)), set_device_ms_min=float(np.min(dev)), set_device_ms_max=float(np.max(dev)),
                set_factor_ms=float(np.median(fac)), set_wall_ms=float(np.median(wall)),
                single_calls_device_ms=sdev, single_calls_wall_ms=swall,
                mean_ir_device_ms=mdev, mean_ir_wall_ms=mwall,
                rel_diff_vs_mean_of_single_calls=float(np.abs(H - ref).max() / np.abs(ref).max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    s = W.params_from_name("WOLA", 256, 16, 8, 10)
    veha = O.synth_channels(250, 21, seed=1)
    rng = np.random.default_rng(1)
    full = (rng.standard_normal((21, 250)) + 1j * rng.standard_normal((21, 250))) * np.exp(-np.arange(21) / 6.0)[:, None]
    res = dict(tool="bench_hessian_set", system="WOLA N=256 cp=16 tails 8/10 (54 variables), L=21", card=card(), reps=a.reps)
    with W.Handle([0]) as h:
        res["veha"] = measure(h, s, veha, a.reps)
        res["full_rank"] = measure(h, s, full, a.reps)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
