"""Bit-for-bit comparison of the BER entry points of two builds of libwofdm.so (the host code of csrc/ber_host.cu).

    python tools/ber_host_ab.py --libs A.so B.so [--out record.json]

Builds nothing.  Runs itself once per library in a fresh process with WOFDM_LIB set to it (capi.load reads it), calls
every wofdm_ber_run* entry point, the plan API and wofdm_ber_verify through the C ABI on fixed seeds, and compares what
the two runs returned: the return code, and every output buffer in full (counters, totals, ensemble_used, rounds;
buffers are filled with a sentinel before each call, so entries a call leaves alone are compared too).  Covered: resolve
0-3 where allowed; shards (0, 1), (1, 3), (46, 47); two window pairs; fp64 jobs, which run the staged kernel, and the
staged resolved twin (WOFDM_RESOLVED_STAGED=1); the channel-mask chain on the mask product and on WOFDM_MASK_FFT=1;
adaptive runs that stop early and ones whose target cannot be reached; and one malformed argument per check of each call
(several where the order of the checks decides the code).  Needs one GPU.  Exit status 1 on any difference.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True

SENTINEL = -7
NOUT = 2 * 4 * 4 * 256            # n_var x n_snr x C x N: the largest output of any call below

ORDER = {   # argument names of each entry point, in the order of include/wofdm.h
    "wofdm_ber_run": "h sys wt wr ch L C snr ns E seed var be bt se st",
    "wofdm_ber_run_shard": "h sys wt wr ch L C snr ns E seed var k W be bt se st",
    "wofdm_ber_run_multi": "h sys wt wr nv ch L C snr ns E seed var k W be bt se st",
    "wofdm_ber_run_resolved": "h sys wt wr nv ch L C snr ns E seed var k W res be se st",
    "wofdm_ber_run_segments": "h sys wt wr nv ch L C snr ns E segs nseg seed var k W res be se st",
    "wofdm_ber_run_adaptive": "h sys wt wr nv ch L C snr ns E fb kind tgt seed var k W red user used be bt se st rounds",
    "wofdm_ber_run_masked": "h sys wt wr ch L C snr ns E seed var ro be bt se st",
    "wofdm_ber_run_masked_shard": "h sys wt wr ch L C snr ns E seed var ro k W be bt se st",
    "wofdm_ber_run_masked_resolved": "h sys wt wr ch L C snr ns E seed var ro k W res be se st",
    "wofdm_ber_run_masked_segments": "h sys wt wr ch L C snr ns E segs nseg seed var ro k W res be se st",
    "wofdm_ber_run_masked_adaptive": "h sys wt wr ch L C snr ns E fb kind tgt seed var ro k W red user used be bt se st rounds",
}
OUTS = ("be", "bt", "se", "st", "used")
SHARDS = ((0, 1), (1, 3), (46, 47))
SEGS = [(2, 2, 3), (0, 0, 2), (1, 4, 1), (1, 2, 2), (2, 0, 2), (0, 2, 3), (1, 0, 1), (1, 1, 1), (3, 1, 4)]


def run_all():
    import wofdm_b200 as W
    from oracle import wofdm_oracle as O
    lib = W.capi.load()
    records = []
    p = O.system_params("wtx", 256, 16, 8, 0, S=16, bits=4, noise_norm=1, constellation=1, guard=64)
    s32 = W.SysT(N=p.N, cp=p.cp, cs=p.cs, tail_tx=p.tail_tx, tail_rx=p.tail_rx, rm=p.rm, shift=p.shift, bits=p.bits, S=p.S,
                 noise_norm=1, constellation=1, precision=0, guard=p.guard)
    s64 = s32.copy(precision=1, S=4)
    bad_guard = s32.copy(bits=8)                            # validate_sys: WOFDM_EUNSUPPORTED
    bad_n = s32.copy(N=100)                                 # validate_sys: WOFDM_EINVAL
    s_n64 = W.params_from_name("CP", 64, 8, 0, 0, bits=4, S=4, noise_norm=1, constellation=1)
    s_long = W.SysT(N=128, cp=80, cs=0, tail_tx=0, tail_rx=0, rm=80, shift=0, bits=4, S=4, noise_norm=1, constellation=1)
    keep = [s32, s64, bad_guard, bad_n, s_n64, s_long]
    wins = [O.perturbed_windows(p, seed=q)[:2] for q in (4, 9)]
    wt = np.ascontiguousarray([w[0] for w in wins], dtype=np.float64)
    wr = np.ascontiguousarray([w[1] for w in wins], dtype=np.float64)
    chans = O.synth_channels(4, 21, seed=5)
    chf = np.ascontiguousarray(chans.T, dtype=np.complex128).view(np.float64)
    snr = np.ascontiguousarray([0.0, 6.0, 12.0, 18.0])
    segs = np.ascontiguousarray(SEGS, dtype=np.int64)
    bufs = {k: np.zeros(NOUT, dtype=np.int64) for k in OUTS}
    rounds = C.c_int(0)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))          # noqa: E731
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))           # noqa: E731
    ident = W.capi.REDUCE_FN(lambda ptr, n, user: 0)               # a reduce over one process: the counts as they are
    nul = W.capi.REDUCE_FN()
    h = W.Handle([0])

    def call(tag, fn, env=None, **over):
        a = dict(h=h._h, sys=C.byref(s32), wt=dp(wt), wr=dp(wr), nv=1, ch=dp(chf), L=21, C=4, snr=dp(snr), ns=4, E=5,
                 segs=ip(segs), nseg=len(SEGS), seed=11, var=1, k=0, W=1, res=0, ro=10, fb=1, kind=1, tgt=50, red=nul,
                 user=None, rounds=C.byref(rounds), **{k: ip(v) for k, v in bufs.items()})
        for k, v in over.items():
            a[k] = C.byref(v) if k == "sys" and v is not None else v
        for b in bufs.values():
            b[:] = SENTINEL
        rounds.value = SENTINEL
        for k, v in (env or {}).items():
            os.environ[k] = v
        try:
            rc = getattr(lib, fn)(*[a[n] for n in ORDER[fn].split()])
        finally:
            for k in env or {}:
                del os.environ[k]
        outs = b"".join(bufs[k].tobytes() for k in OUTS) + rounds.value.to_bytes(4, "little", signed=True)
        rec = dict(id=f"{fn} {tag}", rc=int(rc), outputs=hashlib.sha256(outs).hexdigest()[:16],
                   sym_err=int(bufs["se"][bufs["se"] != SENTINEL].sum()), rounds=rounds.value)
        records.append(rec)
        return rec

    # ---- valid jobs of the main chain: fp32 (tensor-core kernel) and fp64 (staged kernel)
    for prec, s in (("fp32", s32), ("fp64", s64)):
        call(f"{prec}", "wofdm_ber_run", sys=s)
        for k, w in SHARDS:
            call(f"{prec} shard {k}/{w}", "wofdm_ber_run_shard", sys=s, k=k, W=w)
            call(f"{prec} shard {k}/{w} 2 pairs", "wofdm_ber_run_multi", sys=s, nv=2, k=k, W=w)
            for res in (0, 1, 2, 3):
                if res:
                    call(f"{prec} shard {k}/{w} 2 pairs resolve {res}", "wofdm_ber_run_resolved", sys=s, nv=2, k=k, W=w, res=res)
                call(f"{prec} shard {k}/{w} 2 pairs resolve {res}", "wofdm_ber_run_segments", sys=s, nv=2, k=k, W=w, res=res, E=8)
        for nv in (1, 2):
            for kind, tgt, fb in ((1, 50, 1), (0, 400, 2), (1, 10 ** 15, 1), (0, 10 ** 15, 8)):
                call(f"{prec} {nv} pairs kind {kind} target {tgt} first_block {fb}", "wofdm_ber_run_adaptive", sys=s, nv=nv,
                     kind=kind, tgt=tgt, fb=fb, E=8)
            call(f"{prec} {nv} pairs shard 1/3 identity reduce", "wofdm_ber_run_adaptive", sys=s, nv=nv, k=1, W=3, red=ident, E=8)
    staged = {"WOFDM_RESOLVED_STAGED": "1"}
    for res in (1, 3):
        call(f"staged twin resolve {res}", "wofdm_ber_run_resolved", env=staged, nv=2, res=res, k=1, W=3)
        call(f"staged twin resolve {res}", "wofdm_ber_run_segments", env=staged, nv=2, res=res, E=8)

    # ---- valid jobs of the channel-mask chain: the mask product and the per-symbol FFT kernel
    for path, env in (("product", {}), ("fft", {"WOFDM_MASK_FFT": "1"})):
        call(f"{path}", "wofdm_ber_run_masked", env=env)
        for k, w in SHARDS:
            call(f"{path} shard {k}/{w}", "wofdm_ber_run_masked_shard", env=env, k=k, W=w)
            for res in (0, 1, 2, 3):
                if res:
                    call(f"{path} shard {k}/{w} resolve {res}", "wofdm_ber_run_masked_resolved", env=env, k=k, W=w, res=res)
                call(f"{path} shard {k}/{w} resolve {res}", "wofdm_ber_run_masked_segments", env=env, k=k, W=w, res=res, E=8)
        for kind, tgt, fb in ((1, 50, 1), (0, 400, 2), (1, 10 ** 15, 1), (0, 10 ** 15, 8)):
            call(f"{path} kind {kind} target {tgt} first_block {fb}", "wofdm_ber_run_masked_adaptive", env=env, kind=kind,
                 tgt=tgt, fb=fb, E=8)
        call(f"{path} shard 1/3 identity reduce", "wofdm_ber_run_masked_adaptive", env=env, k=1, W=3, red=ident, E=8)

    # ---- one malformed argument per check (and pairs whose order of checks decides the code)
    bad_segs = {"no list": dict(segs=None), "n_seg 0": dict(nseg=0), "overlap": dict(segs=ip(np.ascontiguousarray(
        [(1, 0, 4), (1, 3, 2)], dtype=np.int64)), nseg=2), "outside": dict(segs=ip(np.ascontiguousarray(
            [(4, 0, 1)], dtype=np.int64)), nseg=1), "past ensemble_max": dict(segs=ip(np.ascontiguousarray(
                [(0, 4, 5)], dtype=np.int64)), nseg=1)}
    common = {"handle NULL": dict(h=None), "sys NULL": dict(sys=None), "N 100": dict(sys=bad_n),
              "guard with 256-QAM": dict(sys=bad_guard), "L 0": dict(L=0), "C 0": dict(C=0), "n_snr 0": dict(ns=0),
              "ensemble 0": dict(E=0), "ensemble overflow": dict(E=2 ** 62), "shard -1/2": dict(k=-1, W=2),
              "shard 2/2": dict(k=2, W=2), "shard 0/0": dict(k=0, W=0), "win_tx NULL": dict(wt=None),
              "win_rx NULL": dict(wr=None), "chan NULL": dict(ch=None), "snr NULL": dict(snr=None),
              "bad shard and guard with 256-QAM": dict(k=3, W=2, sys=bad_guard),
              "ensemble 0 and guard with 256-QAM": dict(E=0, sys=bad_guard),
              "win_tx NULL and guard with 256-QAM": dict(wt=None, sys=bad_guard),
              "C 0 and guard with 256-QAM": dict(C=0, sys=bad_guard)}
    masked_only = {"fp64": dict(sys=s64), "N 64": dict(sys=s_n64, wt=dp(np.ones(s_n64.n_tx)), wr=dp(np.ones(64))),
                   "cp + cs too long": dict(sys=s_long, wt=dp(np.ones(s_long.n_tx)), wr=dp(np.ones(128))),
                   "roll_off 0": dict(ro=0), "roll_off too wide": dict(ro=1000),
                   "bad shard and fp64": dict(k=3, W=2, sys=s64), "roll_off 0 and fp64": dict(ro=0, sys=s64),
                   "C 0 and fp64": dict(C=0, sys=s64), "win_tx NULL and fp64": dict(wt=None, sys=s64)}
    for fn, outs in (("wofdm_ber_run", "be bt se st"), ("wofdm_ber_run_shard", "be bt se st"),
                     ("wofdm_ber_run_multi", "be bt se st"), ("wofdm_ber_run_resolved", "be se st"),
                     ("wofdm_ber_run_segments", "be se st"), ("wofdm_ber_run_adaptive", "used be bt se st rounds"),
                     ("wofdm_ber_run_masked", "be bt se st"), ("wofdm_ber_run_masked_shard", "be bt se st"),
                     ("wofdm_ber_run_masked_resolved", "be se st"), ("wofdm_ber_run_masked_segments", "be se st"),
                     ("wofdm_ber_run_masked_adaptive", "used be bt se st rounds")):
        names = ORDER[fn].split()
        base = dict(res=1) if fn.endswith("resolved") else {}
        if "adaptive" in fn:
            base["E"] = 8
        faults = dict(common)
        if "masked" in fn:
            faults.update(masked_only)
        if "nv" in names:
            faults.update({"n_var 0": dict(nv=0), "n_var 9": dict(nv=9)})
        if "res" in names:
            faults.update({"resolve 4": dict(res=4), "resolve -1": dict(res=-1),
                           "resolve 5 and guard with 256-QAM": dict(res=5, sys=bad_guard),
                           "counter array overflow": dict(res=3, ns=1 << 30, C=1 << 30)})
            if fn.endswith("resolved"):
                faults["resolve 0"] = dict(res=0)
        if "segs" in names:
            faults.update(bad_segs)
        if "tgt" in names:
            faults.update({"target_kind 2": dict(kind=2), "target 0": dict(tgt=0), "first_block 0": dict(fb=0),
                           "shard 0/2 without reduce": dict(k=0, W=2), "target 0 and guard with 256-QAM":
                           dict(tgt=0, sys=bad_guard)})
            if "masked" in fn:
                faults["variant too large"] = dict(var=0xfffffff0)
        for o in outs.split():
            faults[f"{o} NULL"] = {o: None}
            faults[f"{o} NULL and guard with 256-QAM"] = {o: None, "sys": bad_guard}
        if fn in ("wofdm_ber_run", "wofdm_ber_run_shard", "wofdm_ber_run_multi", "wofdm_ber_run_resolved"):
            del faults["ensemble overflow"]     # (not rejected before this change: the run's frame count overflowed)
        for tag, over in faults.items():
            call(f"bad: {tag}", fn, **{**base, **over})

    # ---- the plan API (wofdm_ber_plan_read) and the verify path
    for nv in (1, 2):
        plan = C.c_void_p()
        rc = (lib.wofdm_ber_plan_create_multi(h._h, C.byref(s32), dp(wt), dp(wr), nv, dp(chf), 21, 4, dp(snr), 4, C.byref(plan))
              if nv == 2 else lib.wofdm_ber_plan_create(h._h, C.byref(s32), dp(wt), dp(wr), dp(chf), 21, 4, dp(snr), 4,
                                                        C.byref(plan)))
        assert rc == 0, rc
        for k, w in SHARDS:
            be, se = np.full(8, SENTINEL, dtype=np.int64), np.full(8, SENTINEL, dtype=np.int64)
            rc1 = lib.wofdm_ber_plan_launch(plan, 0, 5, 11, 1, k, w, None, None)
            rc2 = lib.wofdm_ber_plan_read(plan, ip(be), ip(se))
            records.append(dict(id=f"wofdm_ber_plan_read {nv} pairs shard {k}/{w}", rc=int(rc1 or rc2),
                                outputs=hashlib.sha256(be.tobytes() + se.tobytes()).hexdigest()[:16], sym_err=int(se.sum())))
        records.append(dict(id=f"wofdm_ber_plan_read {nv} pairs bit_err NULL", rc=int(lib.wofdm_ber_plan_read(plan, None, ip(se)))))
        lib.wofdm_ber_plan_destroy(plan)
    rng = np.random.default_rng(0)
    n = O.noise_len(p, 21)
    sym = rng.integers(0, 16, size=(2, p.S, p.N))
    nz = rng.standard_normal((2, n)) + 1j * rng.standard_normal((2, n))
    for prec, s in (("fp32", s32), ("fp64", s32.copy(precision=1))):
        for kw in ({}, dict(force_staged=True), dict(direct=True)):
            eq, dec, be, se = h.ber_verify(s, wins[0][0], wins[0][1], chans[:, :2], snr[:2], sym, nz, **kw)
            blob = b"".join(np.ascontiguousarray(x).tobytes() for x in (eq, dec, be, se))
            records.append(dict(id=f"wofdm_ber_verify {prec} {sorted(kw)}", rc=0, outputs=hashlib.sha256(blob).hexdigest()[:16],
                                sym_err=int(np.sum(se))))
    h.close()
    del keep
    return records


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--libs", nargs=2, metavar=("A", "B"), help="the two builds of libwofdm.so to compare")
    ap.add_argument("--out", default=None, help="write the comparison record (JSON) here")
    ap.add_argument("--one", default=None, help=argparse.SUPPRESS)     # child process: write this library's results here
    a = ap.parse_args()
    if a.one:
        with open(a.one, "w") as f:
            json.dump(run_all(), f)
        return 0
    if not a.libs:
        ap.error("--libs A B is required")
    runs = []
    for i, lib in enumerate(a.libs):
        tmp = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"ber_host_ab_{os.getpid()}_{i}.json")
        env = dict(os.environ, WOFDM_LIB=os.path.abspath(lib))
        subprocess.run([sys.executable, os.path.abspath(__file__), "--one", tmp], env=env, check=True)
        with open(tmp) as f:
            runs.append(json.load(f))
        os.remove(tmp)
    ra, rb = runs
    diffs = [dict(id=x["id"], a=x, b=y) for x, y in zip(ra, rb) if x != y]
    if len(ra) != len(rb) or [x["id"] for x in ra] != [y["id"] for y in rb]:
        diffs.append(dict(id="(the two runs made different calls)"))
    rec = dict(libs=a.libs, calls=len(ra), valid_calls=sum(1 for x in ra if x["rc"] == 0), differences=len(diffs),
               codes=sorted({x["rc"] for x in ra}), first_differences=diffs[:20], results=ra)
    print(json.dumps({k: v for k, v in rec.items() if k != "results"}))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(rec, f, indent=0)
    return 1 if diffs else 0


if __name__ == "__main__":
    sys.exit(main())
