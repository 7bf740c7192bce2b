#!/usr/bin/env python
"""bench.py -- w-OFDM BER Monte-Carlo throughput (OFDM symbols/s) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (CUDA, libwofdm.so)
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU arm: port of the reference's loop
    torchrun --nproc-per-node N ... bench.py --gpus N ...          # N > 1: one rank per GPU
    python bench.py ... --dump-outputs DIR                         # + the last timed step's counters as DIR/*.npy

A step = one pass of the BER chain over one batch of BASELINE.json configs[1] -- wtx-OFDM, N=256, cp=16, tail_tx=8,
16-QAM, optimised-Tx-window stand-in, the full channel set (250 Vehicular-A realisations, 21 taps), 30 SNR points
linspace(-20,50,30) -- in the reference's PYTHON conventions (the ones its runnable code pins: natural-order
16-QAM, SNR fixed on the truncated signal).  The batch is `--reps` (16) times the 1e8 bits per SNR point of configs[1]
per GPU (ensemble 27 x 16 -> 3.24 M frames = 51.8 M OFDM symbols per GPU and step, one kernel launch), so that the timed
region is seconds, not milliseconds, long.  Weak scaling: the ensemble grows with N, frames are sharded by global frame
id, one all-reduce of the int64 counters per step.
Beside the headline the line carries: `e2e` (host buffers through the C-ABI), `roofline`, `cpu_baseline`, and the
secondary objects `matlab_convention` (the same batch in MATLAB's conventions), `configs4` / `configs4_l84` (N=1024 stress case), `mask_chain`, `k2`
(interference power, configs[3] shapes, fp64 and TF32-split, channels sharded over the ranks) and, for N > 1, `strong`
(the N=1 batch sharded over N GPUs).  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement".
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (it may be read-only)

METRIC = "w-OFDM BER Monte Carlo OFDM symbols/s"
UNIT = "OFDM symbols/s"
# the workload both arms name (the driver compares the strings); everything arm-specific lives in other config keys
WORKLOAD = ("configs[1]: wtx-OFDM N=256 cp=16 tail_tx=8 16-QAM, optimised-Tx-window stand-in, 250 VehA channels x 30 SNR points "
            "linspace(-20,50,30), S=16, L=21, python conventions (natural-order 16-QAM, SNR on the truncated signal), "
            "one window pair per frame")
WORKLOAD4 = ("configs[4]: WOLA-OFDM N=1024 cp=64 tail_tx=32 tail_rx=40 64-QAM, optimised-window stand-ins, 10000 VehA channels "
             "(GMEDS_1, generated on the device) x 30 SNR points, S=16, L=21, python conventions, one window pair per frame")
CFG = dict(system="wtx", N=256, cp=16, tail_tx=8, tail_rx=0, bits=4, S=16, L=21, C=250, n_snr=30,
           snr_lo=-20.0, snr_hi=50.0, ensemble=27, noise_norm=0, constellation=0, name=WORKLOAD)
# BASELINE.json configs[4], the scaled stress case: 1e10 bits per SNR point = ensemble 11 over 10 000 channels
CFG4 = dict(system="WOLA", N=1024, cp=64, tail_tx=32, tail_rx=40, bits=6, S=16, L=21, C=10000, n_snr=30,
            snr_lo=-20.0, snr_hi=50.0, ensemble=11, noise_norm=0, constellation=0, name=WORKLOAD4)
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12          # 74.4: 128 FMA lanes per SM at clocks.max.sm


def workload_inputs(cfg, handle=None):
    """Synthetic inputs of the named shapes (nothing ships with the reference, SURVEY F2).  Pure numpy, except the
    stress workload's 10 000 channels, which come from the device generator (K4) when a handle is given."""
    rng = np.random.default_rng(1)
    L, C = cfg["L"], cfg["C"]
    snr = np.linspace(cfg["snr_lo"], cfg["snr_hi"], cfg["n_snr"])
    if handle is not None and C > 1000:
        fd, fs, frame = (100 / 3.6 / 299792458.0) * 2e9, 5e6, 16 * 256 * 200e-9        # wofdm_optimization.py:63-76
        return handle.gen_channels("vehicularA", L, fd, fs, frame, no_frames=1, n_sets=C, seed=1), snr
    d = np.array([0.0, 310, 710, 1090, 1730, 2510]) / 200.0            # ITU-R VehA delays in samples (Ts = 200 ns)
    pw = 10.0 ** (np.array([0.0, -1, -9, -10, -15, -20]) / 10.0)
    g = (rng.standard_normal((6, C)) + 1j * rng.standard_normal((6, C))) * np.sqrt(pw / 2)[:, None]
    axis = np.arange(L) - (L - 1) / 2.0
    return np.sinc(d[None, :] - axis[:, None]) @ g, snr                # (L, C) complex128


def windows_for(cfg, capi, s):
    """"Optimised" window stand-ins (SURVEY App. B): RC tails perturbed by a seeded +-10 %."""
    rng = np.random.default_rng(7)
    win_tx, win_rx = capi.rc_window_tx(s), capi.rc_window_rx(s)
    if cfg["tail_tx"] > 0:
        x = np.concatenate([[1.0], np.clip(win_tx[-cfg["tail_tx"]:] * (1 + 0.1 * rng.uniform(-1, 1, cfg["tail_tx"])), 0, 1)])
        win_tx = capi.expand_window_tx(s, x)
    return win_tx, win_rx


def flops_per_symbol(N, n_tx, stride, tail_rx, L):
    """SURVEY.md section 8(d): algorithmic real flops per OFDM symbol."""
    f_fft = 2 * 5 * N * int(math.log2(N))
    f_conv = 8 * L * stride
    f_misc = 2 * n_tx + 2 * (N + tail_rx) + 2 * tail_rx + 4 * stride + 8 * stride + 8 * N
    return f_fft, f_conv, f_misc


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
            time.sleep(0.15)                       # first sample before the region starts
        except OSError:
            self.proc = None
        self.t0 = time.time()
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def __exit__(self, *a):
        self.t1 = time.time()
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            self.thr.join(timeout=2)

    def summary(self):
        sm, mx, pw, reasons = [], [], [], set()
        for ts, r in self.rows:
            if ts < self.t0 + 0.1 or ts > self.t1:          # samples taken while the timed region ran
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": float(np.median(pw)), "power_w_max": max(pw)}


_NUMBA_CACHE = None


def cpu_port_throughput(budget_s, workers):
    """The CPU port of the reference's loop (oracle/wofdm_cpu_port.py) on a bounded sample of the workload."""
    global _NUMBA_CACHE
    if "NUMBA_CACHE_DIR" not in os.environ:              # numba would cache the port next to its source, in the tree
        _NUMBA_CACHE = tempfile.TemporaryDirectory(prefix="wofdm_numba_")
        os.environ["NUMBA_CACHE_DIR"] = _NUMBA_CACHE.name
    from oracle import wofdm_cpu_port as P
    c = CFG
    chan, snr = workload_inputs(c)

    def tasks_for(ens, n_tasks, seed0):
        return [P.build_task(c["system"], c["N"], c["cp"], c["tail_tx"], c["tail_rx"], c["S"], c["bits"],
                             chan[:, (k % c["C"]):(k % c["C"]) + 1], ens, snr, seed0 + k) for k in range(n_tasks)]
    # calibrate on one core: 30 SNR points x 1 channel x ensemble 1 = 480 symbols
    rate1, _, _, _ = P.timed_throughput(tasks_for(1, 1, 0), 1)
    n_tasks = max(workers, 1) * 2
    ens = max(1, int(rate1 * budget_s * 0.8 / (c["n_snr"] * c["S"] * 2)))
    val, dt, syms, _ = P.timed_throughput(tasks_for(ens, n_tasks, 100), workers)
    sample = (f"{n_tasks} tasks x ({c['n_snr']} SNR x 1 channel x ensemble {ens}) = {syms} OFDM symbol evaluations of the "
              f"configs[1] workload, ONE window pair per frame (the reference's loop evaluates two, optimised and RC), in {dt:.1f} s; "
              f"numba dense-matrix port of wofdm_simulation.py:171-240, one process per core")
    return val, sample, rate1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workers = os.cpu_count() or 1
    vals = []
    sample = ""
    for i in range(args.warmup + args.steps):
        budget = 2.0 if i < args.warmup else max(3.0, min(12.0, 120.0 / max(args.steps, 1)))
        v, sample, _ = cpu_port_throughput(budget, workers)
        if i >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "note": "CPU arm: every step is a bounded sample of the workload on all host cores, one process per core"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_JSON_FD = None


def emit(line):
    """The one JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


class Job:
    """One BER workload on this rank's GPU: plan + timed launches (device-resident inputs)."""

    def __init__(self, torch, dist, W, capi, h, cfg, world, rank, reps, scaling="weak"):
        self.torch, self.dist, self.h, self.cfg, self.world, self.rank = torch, dist, h, cfg, world, rank
        c = cfg
        self.s = W.params_from_name(c["system"], c["N"], c["cp"], c["tail_tx"], c["tail_rx"], bits=c["bits"], S=c["S"],
                                    noise_norm=c["noise_norm"], constellation=c["constellation"], precision=0)
        self.win_tx, self.win_rx = windows_for(c, capi, self.s)
        self.chan, self.snr = workload_inputs(c, h)
        ens_gpu = c["ensemble"] * reps
        # weak: every GPU adds its own ensemble; strong: the one-GPU batch is shared out
        self.ens_total = ens_gpu * world if scaling == "weak" else ens_gpu
        self.shard = (rank, world)
        total = c["n_snr"] * c["C"] * self.ens_total
        self.frames_rank = (total - rank + world - 1) // world
        self.frames_job = total
        self.plan = h.ber_plan(self.s, self.win_tx, self.win_rx, self.chan, self.snr)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, stream, flush, steps, warmup, seed0, clocks=None):
        """-> (ms of the whole region as the max over ranks, mean kernel ms, mean all-reduce ms)"""
        torch, dist, c = self.torch, self.dist, self.cfg
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
        with torch.cuda.stream(stream):
            for i in range(warmup):
                self.plan.launch(self.ens_total, seed=seed0 + i, shard=self.shard, stream=stream.cuda_stream)
            self.barrier()
            ctx = clocks if clocks is not None else _Null()
            with ctx:
                for i in range(steps):
                    flush.fill_(i & 0xff)                                       # evict L2 between timed iterations
                    ev[i][0].record(stream)
                    dptr = self.plan.launch(self.ens_total, seed=seed0 + 100 + i, shard=self.shard, stream=stream.cuda_stream)
                    ev[i][1].record(stream)
                    if self.world > 1:                                          # the path's only exchange step
                        dist.all_reduce(_as_tensor(torch, dptr, c["n_snr"] * 2))
                    ev[i][2].record(stream)
                self.barrier()
        ms_rank = sum(e[0].elapsed_time(e[2]) for e in ev)
        kms = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
        ams = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
        t = torch.tensor([ms_rank], dtype=torch.float64, device="cuda")
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), kms, ams

    def symbols_job(self):
        return self.frames_job * self.cfg["S"]

    def roofline_tflops(self, kms):
        f = flops_per_symbol(self.s.N, self.s.n_tx, self.s.stride, self.s.tail_rx, self.cfg["L"])
        return sum(f) * self.frames_rank * self.cfg["S"] / (kms * 1e-3) / 1e12, f


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def gemm_peaks(torch):
    """cuBLAS GEMM rates measured in this process: the flop-based denominators of the interference GEMMs."""
    out = {}
    for key, dt, n, tf32 in (("fp64_tflops", torch.float64, 4096, False), ("tf32_tflops", torch.float32, 8192, True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        a = torch.randn(n, n, dtype=dt, device="cuda")
        b = torch.randn(n, n, dtype=dt, device="cuda")
        for _ in range(2):
            torch.matmul(a, b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b); e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        out[key] = 2.0 * n ** 3 / (best * 1e-3) / 1e12
        del a, b
    torch.backends.cuda.matmul.allow_tf32 = False
    return out


def k2_section(torch, dist, W, capi, h, world, rank):
    """Interference power (BASELINE configs[3] shapes: WOLA N=256 cp=16, 250 channels, M = 2 slices), through the C-ABI
    with host buffers.  N > 1: the channel realisations are sharded in contiguous blocks and the per-channel rows meet
    in one NCCL all-gather inside the timed call (sharding.allgather_channel_rows)."""
    from wofdm_b200 import sharding
    s = W.params_from_name("WOLA", 256, 16, 8, 10, precision=1)
    vt, vr = capi.rc_window_tx(s), capi.rc_window_rx(s)
    chan, _ = workload_inputs(dict(L=21, C=250, snr_lo=0, snr_hi=1, n_snr=1))
    lo, hi = sharding.channel_block(chan.shape[1], rank, world)
    mine = np.ascontiguousarray(chan[:, lo:hi])
    n_rx, n_tx, N = s.stride, s.n_tx, s.N
    M = 1 + -(-(21 - 1 + s.tail_tx) // n_rx)
    dense = (8 * N * n_rx * n_tx + 8 * N * n_tx * N) * chan.shape[1] * M          # SURVEY 8(d): per (channel, slice)
    out = {"shapes": f"WOLA N=256 cp=16: Rx_mat {N}x{n_rx}, H {n_rx}x{n_tx}, Tx_mat {n_tx}x{N}, {chan.shape[1]} channels x {M} slices",
           "dense_gflop_per_call": dense / 1e9,
           "api": "wofdm_interf_power (ctypes, host buffers in, per-channel rows out)"}
    for mode, key in ((0, "fp64"), (1, "tf32"), (2, "quad")):
        for _ in range(3):
            P = h.interf_power(s, vt, vr, mine, mode=mode)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        reps, t_g = 10, 0.0
        t0 = time.perf_counter()
        for _ in range(reps):
            P = h.interf_power(s, vt, vr, mine, mode=mode)
            if world > 1:
                g0 = time.perf_counter()
                allP = sharding.allgather_channel_rows(torch.from_numpy(P).cuda(), chan.shape[1])
                torch.cuda.synchronize()
                t_g += time.perf_counter() - g0
        dt = (time.perf_counter() - t0) / reps
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            assert allP.shape[0] == chan.shape[1]
        dt = float(t.item())
        tm = h.interf_last_timing()
        # executed tensor-core GEMM: slice 0 contracts all K rows, an ISI slice only its non-zero prefix
        # (mode 2, "quad": the contraction runs on the L unit-impulse channels, every realisation is a Hermitian form in its taps)
        gemm = 2 * (2 * N) * (tm["k_slice0"] + (M - 1) * tm["k_isi"]) * N * (21 if mode == 2 else mine.shape[1])
        out[key + "_ms"] = dt * 1e3
        out[key + "_device_ms"], out[key + "_band_product_ms"], out[key + "_gemm_ms"] = tm["total_ms"], tm["band_ms"], tm["gemm_ms"]
        out[key + "_dense_tflops"] = dense / dt / 1e12
        out[key + "_executed_gflop_per_rank"] = gemm / 1e9
        out[key + "_gemm_kernel_tflops"] = gemm / (tm["gemm_ms"] * 1e-3) / 1e12 if tm["gemm_ms"] > 0 else None
        out[key + "_executed_tflops"] = gemm / dt / 1e12
        if world > 1:
            out[key + "_allgather_ms"] = t_g / reps * 1e3
        out[key + "_p_total"] = float(P.sum())
    out["quad_note"] = ("mode 2: fp64 like mode 0 (results agree to ~1e-14), but A_m(c) = sum_l h_c[l] G_{m,l}: the L = 21 impulse "
                        "responses go through the mode-0 band product and DMMA contraction once per window pair, then every "
                        "channel is P_k = h^H Q_k h (one C x L(L+1) x N real product); quad_executed_* count those 21 slices' GEMM")
    out["quad_speedup_vs_fp64"] = out["fp64_ms"] / out["quad_ms"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary objects (matlab_convention, configs4, k2, strong)")
    ap.add_argument("--reps", type=int, default=16, help="multiples of configs[1]'s 1e8 bits per SNR point per GPU and step")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default): per-GPU work fixed; strong: the one-GPU batch sharded over the GPUs")
    ap.add_argument("--workload", default="configs1", choices=["configs1", "configs4"],
                    help="configs1 = BASELINE's headline configuration (default); configs4 = the N=1024 stress case")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the counters of the last timed step (bit_err, bit_tot, sym_err, sym_tot per SNR point) "
                         "as DIR/<name>.npy, float64, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the CPU arm times a sample of the workload, not the timed GPU path")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    cfg = dict(CFG)
    if args.workload == "configs4":
        cfg = dict(CFG4)
        args.no_cpu_baseline = True          # the CPU port is dimensioned for the headline workload
        args.reps = 1

    # stdout carries ONE JSON line: NCCL writes its log lines to stdout by default ("NCCL version ..." was seen on the
    # multi-GPU boxes, where NCCL_DEBUG=VERSION ignores NCCL_DEBUG_FILE), so every other writer of file descriptor 1 --
    # C libraries included -- is sent to stderr and the JSON line goes out through the saved descriptor
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    import wofdm_b200 as W
    from wofdm_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} needs WORLD_SIZE={args.gpus} (launch with torch.distributed.run); got {world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    h = W.Handle([local])
    stream = torch.cuda.Stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    peak_tflops, peak_mhz = h.fp32_peak(0)

    # ---------------- device-resident arm: inputs live in HBM, one kernel launch per step ----------------
    job = Job(torch, dist, W, capi, h, cfg, world, rank, args.reps, args.scaling)
    c, s = cfg, job.s
    launches0 = h.launches
    clocks = ClockSampler(local)
    ms_total, kms, ams = job.timed(stream, flush, args.steps, args.warmup, 1000, clocks)
    launches = h.launches - launches0 - args.warmup
    value = job.symbols_job() * args.steps / (ms_total * 1e-3)
    be, se = job.plan.read()
    bt, st_ = job.plan.totals(job.ens_total, job.shard if world == 1 else (0, 1))
    # (N > 1: the in-place all-reduce left the job-wide counters in every rank's device buffer)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in (("bit_err", be), ("bit_tot", bt), ("sym_err", se), ("sym_tot", st_)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(a, dtype=np.float64))   # exact below 2**53

    # ---------------- end-to-end arm: C-ABI call with HOST buffers, copies inside the timed region ----------------
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    win_tx_p, win_rx_p, chan_p, snr_p = pin(job.win_tx), pin(job.win_rx), pin(job.chan), pin(job.snr)
    for i in range(2):
        h.ber_run(s, win_tx_p, win_rx_p, chan_p, snr_p, job.ens_total, seed=3000 + i, shard=job.shard)
    job.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        r = h.ber_run(s, win_tx_p, win_rx_p, chan_p, snr_p, job.ens_total, seed=4000 + i, shard=job.shard)
        if world > 1:
            t = torch.from_numpy(np.stack([r["bit_err"], r["sym_err"]])).cuda()
            dist.all_reduce(t)
            t.cpu()
    torch.cuda.synchronize()
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = job.symbols_job() * args.steps / float(e2e_t.item())
    h2d = (s.n_tx + s.N + s.tail_rx) * 8 + job.chan.size * 16 + job.snr.size * 8
    d2h = c["n_snr"] * 2 * 8

    line = None
    if rank == 0:
        achieved, (f_fft, f_conv, f_misc) = job.roofline_tflops(kms)
        f_chain = f_fft + f_conv + f_misc
        traffic, tsrc = None, None
        tpath = os.path.join(REPO, "profiles", "k1_traffic.json")
        if os.path.exists(tpath) and args.workload == "configs1":
            with open(tpath) as fh:
                tj = json.load(fh)
            traffic, tsrc = tj.get("dram_bytes_per_launch"), tj.get("source")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": c["name"],
                       "batch": f"ensemble {c['ensemble']} x {args.reps} per GPU = {job.frames_rank} frames = "
                                f"{job.frames_rank * c['S']:.4g} OFDM symbols per GPU and step "
                                f"({args.reps} x the {'1e8' if args.workload == 'configs1' else '1e10'} bits per SNR point of the named config), one kernel launch",
                       "kernel": job.plan.kernel, "frames_per_gpu_per_step": job.frames_rank,
                       "l2": "256 MiB buffer rewritten between timed iterations (inputs are ~100 KB; the kernel is FP32-bound)",
                       "parallelism": f"frames sharded by global id over {world} GPU(s), one int64 all-reduce per step"},
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "wofdm_ber_run_shard (ctypes, pinned host buffers in, int64 counters out)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s", "frac": achieved / peak_tflops,
                         "frac_nominal": achieved / NOMINAL_FP32_TFLOPS, "peak_nominal": NOMINAL_FP32_TFLOPS,
                         "traffic": traffic,
                         "traffic_source": tsrc or "not measured in this run (ncu captures: profiles/)",
                         "peak_source": f"FMA-only micro-benchmark run in this process (wofdm_diag_fp32_peak, scalar FFMA): {peak_tflops:.1f} TFLOP/s "
                                        f"= 128 FMA lanes x 148 SMs at {peak_mhz:.0f} MHz; "
                                        "MEASURED_PEAKS.json has no FP32 entry (HBM/bf16 only); frac_nominal is against 74.4 TFLOP/s",
                         "flops_per_symbol": {"fft": f_fft, "conv": f_conv, "misc": f_misc, "chain": f_chain},
                         "kernel_ms": kms, "allreduce_ms": ams if world > 1 else 0.0,
                         "achieved_fft_only": f_fft * job.frames_rank * c["S"] / (kms * 1e-3) / 1e12,
                         "hbm_note": "HBM traffic ~0 (counters only): 'hbm'/'tensor' do not bound this kernel",
                         "bound_note": "on-chip bound: the denominator is the FP32 FMA peak the north star names; the kernel's real "
                                       "limits are the math dispatch port (FFMA2/IMAD/LOP3 = 2 cycles per warp instruction, no "
                                       "co-issue of integer work with packed FP32), shared-memory wavefronts and the barrier skew of "
                                       "16 warps per SM -- DESIGN.md section 3, tools/ubench/pipes*.cu",
                         "tensor_note": ("kernel ber_f32t*: the 'conv' share of the algorithmic flops (the L-tap channel convolution) "
                                         "runs on the tensor pipe (tcgen05 kind::f16, 3-term fp16 split = fp32-grade, DESIGN.md section 3) "
                                         "to relieve the FP32 dispatch port; FFTs, windows, noise, equaliser and slicer stay on the FP32 pipe; "
                                         "the figure is still algorithmic flops / time against the FP32 FMA peak"
                                         if "f32t" in job.plan.kernel else "all arithmetic on the FP32 pipe")},
            "ber_check": {"snr_db": [float(job.snr[k]) for k in (0, 10, 15, 20, 29)],
                          "ser": [float(se[k] / st_[k]) for k in (0, 10, 15, 20, 29)],
                          "ber": [float(be[k] / bt[k]) for k in (0, 10, 15, 20, 29)]},
        }
    job.plan.close()

    # ---------------- secondary objects ----------------
    extras = {}
    if not args.no_extras and args.workload == "configs1":
        steps2 = max(3, min(5, args.steps))
        # (1) the same batch in MATLAB's conventions (Gray unit-power 16-QAM, SNR on the full convolution): parity unpinned
        jm = Job(torch, dist, W, capi, h, dict(CFG, noise_norm=1, constellation=1), world, rank, args.reps, args.scaling)
        ms_m, kms_m, _ = jm.timed(stream, flush, steps2, 3, 5000)
        extras["matlab_convention"] = {"value": jm.symbols_job() * steps2 / (ms_m * 1e-3), "unit": UNIT, "ms_per_step": ms_m / steps2,
                                       "kernel": jm.plan.kernel, "frac": jm.roofline_tflops(kms_m)[0] / peak_tflops,
                                       "note": "noise_norm=1, constellation=1 (main_BER_calculation.m); parity unpinned (no MATLAB/Octave)"}
        jm.plan.close()
        # (2) BASELINE configs[4]: N=1024 stress case, 10 000 channels generated on the device, 1e10 bits per SNR point per GPU
        j4 = Job(torch, dist, W, capi, h, dict(CFG4), world, rank, 1, args.scaling)
        ms_4, kms_4, _ = j4.timed(stream, flush, 3, 3, 6000)
        a4, f4 = j4.roofline_tflops(kms_4)
        extras["configs4"] = {"value": j4.symbols_job() * 3 / (ms_4 * 1e-3), "unit": UNIT, "ms_per_step": ms_4 / 3, "steps": 3,
                              "workload": WORKLOAD4, "kernel": j4.plan.kernel, "frames_per_gpu_per_step": j4.frames_rank,
                              "frac": a4 / peak_tflops, "achieved_tflops": a4, "flops_per_symbol": sum(f4)}
        j4.plan.close()
        # (2b) the same with the 84-tap channels configs[4] names as its option ("L = 21 (optionally 84)")
        j84 = Job(torch, dist, W, capi, h, dict(CFG4, L=84, name=WORKLOAD4.replace("L=21", "L=84")), world, rank, 1, args.scaling)
        ms_8, kms_8, _ = j84.timed(stream, flush, 3, 3, 6500)
        a8, f8 = j84.roofline_tflops(kms_8)
        extras["configs4_l84"] = {"value": j84.symbols_job() * 3 / (ms_8 * 1e-3), "unit": UNIT, "ms_per_step": ms_8 / 3, "steps": 3,
                                  "workload": WORKLOAD4.replace("L=21", "L=84"), "kernel": j84.plan.kernel,
                                  "frac": a8 / peak_tflops, "achieved_tflops": a8, "flops_per_symbol": sum(f8)}
        j84.plan.close()
        # (3) strong scaling: the one-GPU batch sharded over the GPUs (N = 1: identical to the headline, skipped)
        if world > 1 and args.scaling == "weak":
            js = Job(torch, dist, W, capi, h, dict(CFG), world, rank, args.reps, "strong")
            ms_s, kms_s, ams_s = js.timed(stream, flush, steps2, 3, 7000)
            extras["strong"] = {"value": js.symbols_job() * steps2 / (ms_s * 1e-3), "unit": UNIT, "ms_per_step": ms_s / steps2,
                                "kernel_ms": kms_s, "allreduce_ms": ams_s, "allreduce_share": ams_s / (ms_s / steps2),
                                "frames_per_gpu_per_step": js.frames_rank,
                                "note": "fixed total batch (the N=1 headline batch) sharded over the GPUs"}
            js.plan.close()
        # (4) interference power, configs[3] shapes, fp64 and TF32-split, channels sharded over the ranks
        k2 = k2_section(torch, dist, W, capi, h, world, rank)
        if rank == 0:
            pk = gemm_peaks(torch)
            k2.update(pk)
            k2["frac_fp64"] = k2["fp64_gemm_kernel_tflops"] / pk["fp64_tflops"]
            k2["frac_tf32"] = 3.0 * k2["tf32_gemm_kernel_tflops"] / pk["tf32_tflops"]
            k2["frac_fp64_whole_call"] = k2["fp64_executed_tflops"] * world / pk["fp64_tflops"]
            k2["frac_tf32_whole_call"] = 3.0 * k2["tf32_executed_tflops"] * world / pk["tf32_tflops"]
            k2["frac_note"] = ("frac_*: executed tensor-core GEMM flops (slice 0: all K rows; ISI slices: their non-zero K prefix) over "
                               "the contraction kernel's device time (CUDA events inside the library, wofdm_interf_last_timing), against "
                               "the cuBLAS GEMM rate measured in this process (DGEMM 4096^3; TF32 8192^3); the TF32 path executes 3 "
                               "products per fp64 one (3xTF32 split), hence the factor 3.  frac_*_whole_call: the same flops over the "
                               "wall time of the host-buffer call (uploads, matrix builders, band product, download included)")
            tp = os.path.join(REPO, "profiles", "k2_traffic.json")
            if os.path.exists(tp):
                with open(tp) as fh:
                    k2["traffic"] = json.load(fh)
        extras["k2"] = k2
        # (5) the channel-mask BER variant (matlab/main_channel_mask.m; SURVEY 8f-1): guard band N/4 + DFT-domain RC mask, the mask as a
        #     dense tcgen05 product.  One device per call: every rank runs the same call, rank 0 reports its own wall time.
        import time as _time
        import numpy as _np
        sm_ = W.params_from_name("wtx", 256, 16, 8, 0, bits=4, S=16, noise_norm=1, constellation=1, guard=64)
        rng_ = _np.random.default_rng(0)
        ch_ = (rng_.standard_normal((21, 250)) + 1j * rng_.standard_normal((21, 250))) * _np.exp(-_np.arange(21) / 4)[:, None]
        snr_ = _np.linspace(-20, 50, 30)
        vt_, vr_ = capi.rc_window_tx(sm_), capi.rc_window_rx(sm_)
        ens_ = 16
        for _ in range(2):
            h.ber_run_masked(sm_, vt_, vr_, ch_, snr_, ens_, seed=1, variant=1)
        t0_ = _time.perf_counter()
        for k_ in range(3):
            rm_ = h.ber_run_masked(sm_, vt_, vr_, ch_, snr_, ens_, seed=2 + k_, variant=1)
        dt_ = (_time.perf_counter() - t0_) / 3
        extras["mask_chain"] = {"value": 30 * 250 * ens_ * 16 / dt_, "unit": UNIT, "ms_per_call": dt_ * 1e3, "frames_per_call": 30 * 250 * ens_,
                                "api": "wofdm_ber_run_masked (ctypes, host buffers in, int64 counters out; wall time)",
                                "workload": "main_channel_mask.m run_sim_mc: wtx N=256 cp=16 tail_tx=8 16-QAM, 128 active sub-carriers (guard 64), "
                                            "RC mask roll-off 10 bins, 250 channels x 30 SNR points x ensemble 16, MATLAB conventions (parity unpinned)",
                                "ber": [float(rm_["bit_err"][k] / rm_["bit_tot"][k]) for k in (0, 10, 15, 20, 29)]}
    if rank == 0:
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            v, sample, rate1 = cpu_port_throughput(12.0, os.cpu_count() or 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port", "sample": sample,
                                    "single_core": rate1}
        emit(line)
    h.close()
    if world > 1:
        dist.destroy_process_group()


def _as_tensor(torch, dptr, n):
    """int64 view of the library's device counters (no copy) for the NCCL all-reduce."""
    class _Arr:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (int(dptr), False), "version": 3}
    return torch.as_tensor(_Arr(), device="cuda")


if __name__ == "__main__":
    main()
