"""Device time of the N = 1024 tensor-core K1 launch (ber_tconv2.cuh, 2-CTA cluster) in two builds of libwofdm.so, alternated
in one process: the rotation of its MMA-issuing warps keyed on the CTA (before) or on the frame (after) changes nothing else.

bench.py's configs[4] system (WOLA, N = 1024, cp 64, tails 32 / 40, 64-QAM, S = 16), 30 SNR points from -20 to 50 dB, one
window pair, L = 21 and L = 84 taps, frame steps 1 and 8 (shard (0, 1) and (0, 8), the step of an 8-GPU strong-scaling rank:
a CTA's consecutive frames lie nslots * step apart).  Both steps launch the same number of frames.  Each launch is timed with
CUDA events on one stream, the libraries alternate launch by launch in --reps rounds of --launches each, after warm-up.
Reports the median per library and case, the run-to-run spread (min / max of the per-round medians), the counters of both
builds, and the card's name and power limit read in the same run.  One JSON line on stdout (and in --out).

    python tools/bench_ber_n1024_rotation.py --lib before=/path/libwofdm.so --lib after=/path/libwofdm.so"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))
sys.dont_write_bytecode = True
import wofdm_b200 as W  # noqa: E402
from wofdm_b200 import capi  # noqa: E402
from bench import CFG4  # noqa: E402
from bench_ber_resolved import card  # noqa: E402
from oracle import wofdm_oracle as O  # noqa: E402


def open_lib(path):
    lib = ctypes.CDLL(path)
    for name, (res, args) in capi.SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lib", action="append", required=True, help="label=path of a libwofdm.so build (two or more)")
    ap.add_argument("--channels", type=int, default=150, help="channels of the job (configs[4] has 10 000)")
    ap.add_argument("--ensemble", type=int, default=11, help="ensemble at frame step 1 (step k launches k times as many)")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--launches", type=int, default=5, help="launches per library and round")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    libs = dict(x.split("=", 1) for x in a.lib)
    info = card()
    c = CFG4
    s = W.params_from_name(c["system"], c["N"], c["cp"], c["tail_tx"], c["tail_rx"], bits=c["bits"], S=c["S"],
                           noise_norm=c["noise_norm"], constellation=c["constellation"])
    snr = np.linspace(c["snr_lo"], c["snr_hi"], c["n_snr"])
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    stream = torch.cuda.Stream()
    handles, cases = {}, []
    loaded = {k: open_lib(p) for k, p in libs.items()}
    try:
        for k in libs:
            capi._lib = loaded[k]
            handles[k] = W.Handle([0])
        for L in (21, 84):
            chan = O.synth_channels(a.channels, L, seed=L)
            for step in (1, 8):
                ens = a.ensemble * step
                frames = len(snr) * a.channels * ens // step
                plans, kernel, counters = {}, {}, {}
                for k in libs:
                    capi._lib = loaded[k]
                    plans[k] = handles[k].ber_plan(s, vt, vr, chan, snr)
                    kernel[k] = plans[k].kernel

                def launch(k):
                    capi._lib = loaded[k]
                    plans[k].launch(ens, seed=1, shard=(0, step), stream=stream.cuda_stream)

                for k in libs:                                    # warm-up, and the counters of each build
                    for _ in range(2):
                        launch(k)
                    stream.synchronize()
                    capi._lib = loaded[k]
                    be, se = plans[k].read()
                    counters[k] = dict(bit_err=int(be.sum()), sym_err=int(se.sum()))
                rounds = {k: [] for k in libs}
                order = list(libs)
                for r in range(a.reps):
                    for k in (order if r % 2 == 0 else order[::-1]):
                        ms = []
                        for _ in range(a.launches):
                            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            e0.record(stream)
                            launch(k)
                            e1.record(stream)
                            e1.synchronize()
                            ms.append(e0.elapsed_time(e1))
                        rounds[k].append(float(np.median(ms)))
                for k in libs:
                    capi._lib = loaded[k]
                    plans[k].read()
                    plans[k].close()
                res = {}
                for k, t in rounds.items():
                    med = float(np.median(t))
                    res[k] = dict(kernel=kernel[k], median_ms=round(med, 4), min_ms=round(min(t), 4), max_ms=round(max(t), 4),
                                  spread=round((max(t) - min(t)) / med, 4), ofdm_symbols_per_s=round(frames * c["S"] / med * 1e3, 1),
                                  counters=counters[k])
                cases.append(dict(L=L, frame_step=step, frames_per_launch=frames, libs=res))
                print(json.dumps(cases[-1]), file=sys.stderr)
    finally:
        for k, h in handles.items():
            capi._lib = loaded[k]
            h.close()
    rec = dict(metric="device time of one N = 1024 tensor-core K1 launch (CUDA events), builds alternated", card=info,
               workload=f"configs[4] system (WOLA N=1024, 64-QAM, S=16), {a.channels} channels, {len(snr)} SNR points, one window pair",
               timing=f"median over {a.reps} alternated rounds of the per-round median of {a.launches} launches", libs=libs,
               cases=cases)
    line = json.dumps(rec)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
