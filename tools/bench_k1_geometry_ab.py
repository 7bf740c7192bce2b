"""A/B of the K1 kernels at bench.py's headline: the fixed-geometry instance against the class-only loop and the generic kernel.

Every arm is a separate process (the library is loaded once per process), and the arms alternate round by round:
  parent    bench.py with WOFDM_LIB = a build of the parent commit (its "_hs" entry is the class-only loop)
  geometry  bench.py with this tree's library: "_hs" = the loop with the headline geometry compiled in (ber_tconv2.cuh)
  class     the same library, WOFDM_VARIANT=_hsc: the class-only loop (same code as the parent's "_hs")
  generic   the same library, WOFDM_VARIANT=..._tiles9_b2$: the generic kernel
bench.py runs as `--no-extras --steps 20`; the MATLAB-convention batch (bench.py's matlab_convention) is timed with bench's
own Job in a child process per arm.  Finally bench.py --dump-outputs of parent and geometry with the same seeds.
Nothing is compiled at run time: the parent library is built beforehand.

usage: bench_k1_geometry_ab.py --parent-lib PATH [--rounds 3] [--out DIR]   (the tree is only read: results go to DIR)"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GENERIC = "ber_f32t2_n256_t256_tiles9_b2$"


def matlab_child(steps):
    """time bench.py's MATLAB-convention batch exactly as bench.py does (one Job, L2 flushed between steps)"""
    sys.path.insert(0, REPO)
    import torch
    import torch.distributed as dist
    import bench
    import wofdm_b200 as W
    from wofdm_b200 import capi
    torch.cuda.set_device(0)
    h = W.Handle([0])
    stream = torch.cuda.Stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    jm = bench.Job(torch, dist, W, capi, h, dict(bench.CFG, noise_norm=1, constellation=1), 1, 0, 16)
    ms, kms, _ = jm.timed(stream, flush, steps, 3, 5000)
    print(json.dumps({"value": jm.symbols_job() * steps / (ms * 1e-3), "ms_per_step": ms / steps, "kernel_ms": kms,
                      "kernel": jm.plan.kernel}))
    jm.plan.close()
    h.close()


def env_for(arm, parent_lib):
    env = dict(os.environ)
    for k in ("WOFDM_LIB", "WOFDM_VARIANT"):
        env.pop(k, None)
    if arm == "parent":
        env["WOFDM_LIB"] = parent_lib
    elif arm == "class":
        env["WOFDM_VARIANT"] = "_hsc"
    elif arm == "generic":
        env["WOFDM_VARIANT"] = GENERIC
    return env


def last_json(out):
    return json.loads([l for l in out.splitlines() if l.startswith("{")][-1])


def run(cmd, env, log):
    r = subprocess.run(cmd, cwd=REPO, env=env, capture_output=True, text=True, timeout=900)
    log.write(f"$ {' '.join(cmd)}  [{env.get('WOFDM_LIB', '')} {env.get('WOFDM_VARIANT', '')}] rc={r.returncode}\n{r.stderr[-3000:]}\n")
    log.flush()
    if r.returncode != 0:
        raise SystemExit(f"{cmd} failed: {r.stderr[-3000:]}")
    return last_json(r.stdout)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory of the record, the log and the counter dumps (default: a new temporary one)")
    ap.add_argument("--matlab-child", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.matlab_child:
        return matlab_child(args.matlab_child)
    if not os.path.exists(args.parent_lib):
        raise SystemExit(f"no parent library at {args.parent_lib}")
    if args.out is None:
        args.out = tempfile.mkdtemp(prefix="k1_geometry_ab_")
    os.makedirs(args.out, exist_ok=True)
    print(f"output: {args.out}", flush=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    rec = {"gpu": q, "started": time.strftime("%Y-%m-%d %H:%M:%S"), "bench": "bench.py --gpus 1 --no-extras --steps 20 --warmup 3",
           "arms": {}, "matlab": {}}
    log = open(os.path.join(args.out, "k1_geometry_ab.log"), "w")
    bench = [sys.executable, "bench.py", "--gpus", "1", "--no-extras", "--no-cpu-baseline", "--steps", "20", "--warmup", "3"]
    arms = ("parent", "geometry", "class", "generic")
    for rnd in range(args.rounds):
        for arm in (arms if rnd % 2 == 0 else arms[::-1]):
            j = run(bench, env_for(arm, args.parent_lib), log)
            rec["arms"].setdefault(arm, []).append({"value": j["value"], "ms_per_step": j["ms_per_step"],
                                                    "kernel_ms": j["roofline"]["kernel_ms"], "kernel": j["config"]["kernel"],
                                                    "clocks": j.get("clocks")})
            print(f"round {rnd} {arm:8s} {j['value']:.4e} symbols/s  {j['config']['kernel']}", flush=True)
        for arm in (("parent", "geometry") if rnd % 2 == 0 else ("geometry", "parent")):
            j = run([sys.executable, os.path.abspath(__file__), "--parent-lib", args.parent_lib, "--matlab-child", "20"],
                    env_for(arm, args.parent_lib), log)
            rec["matlab"].setdefault(arm, []).append(j)
            print(f"round {rnd} matlab {arm:8s} {j['value']:.4e} symbols/s  {j['kernel']}", flush=True)
    summ = {}
    for key, d in (("headline", rec["arms"]), ("matlab_convention", rec["matlab"])):
        for arm, xs in d.items():
            v = [x["value"] for x in xs]
            summ[f"{key}/{arm}"] = {"mean": sum(v) / len(v), "min": min(v), "max": max(v), "spread": max(v) - min(v)}
    for key in ("headline", "matlab_convention"):
        p, g = summ.get(f"{key}/parent"), summ.get(f"{key}/geometry")
        if p and g:
            summ[f"{key}/geometry_vs_parent"] = g["mean"] / p["mean"] - 1.0
    c, g = summ.get("headline/class"), summ.get("headline/generic")
    if c and g:
        summ["headline/class_vs_generic"] = c["mean"] / g["mean"] - 1.0
    rec["summary"] = summ
    # counters of the same seeds through both libraries
    dumps = {}
    for arm in ("parent", "geometry"):
        d = os.path.join(args.out, f"dump_{arm}")
        run(bench + ["--dump-outputs", d], env_for(arm, args.parent_lib), log)
        dumps[arm] = {n: open(os.path.join(d, n + ".npy"), "rb").read() for n in ("bit_err", "bit_tot", "sym_err", "sym_tot")}
    rec["dump_outputs_identical"] = all(dumps["parent"][n] == dumps["geometry"][n] for n in dumps["parent"])
    print(json.dumps(summ, indent=1))
    print("dump_outputs_identical", rec["dump_outputs_identical"])
    with open(os.path.join(args.out, "k1_geometry_ab.json"), "w") as fh:
        json.dump(rec, fh, indent=1)


if __name__ == "__main__":
    main()
