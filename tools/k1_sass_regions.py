"""SASS instructions of a K1 tensor-core kernel between its barriers, and the two counts its schedule depends on.

The working warps of ber_tconv2.cuh announce their part of the split stream (bar.arrive, SASS BAR.ARV) and then draw their
noise while the MMA warp issues; the accumulator pass waits on the MMAs' mbarrier (SYNCS.PHASECHK).  Draws that ptxas hoists
in front of the arrive delay the MMAs of the whole CTA (DESIGN section 7, constant switches), and the counters do not show
it.  This prints, per kernel, the instructions from the barrier before the arrive to the arrive ("tx->arrive") and from the
arrive to the first wait behind it ("arrive->wait"): production N = 256 and the HS instances have ~25-110 and ~550-650, a
build whose draws were hoisted had 468 and 233.  "frame loop" is the longest backward branch's span (the working warps'
loop over frames); --opcodes adds its instructions by opcode.
usage: k1_sass_regions.py <object or cubin> [kernel-name substring] [--regions] [--opcodes]"""
import collections
import re
import subprocess
import sys


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    fns, cur = {}, None
    for l in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", l)
        if m:
            cur = fns.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", l)
        if m and cur is not None:
            cur.append(re.sub(r"^@!?U?P\w+\s+", "", m.group(1)))
    return fns


def counts(ins):
    arv = [i for i, s in enumerate(ins) if s.startswith("BAR.ARV")]
    if not arv:
        return None
    a = arv[0]
    before = max((i for i in range(a) if ins[i].startswith("BAR.")), default=0)
    wait = next((i for i in range(a, len(ins)) if ins[i].startswith("SYNCS.PHASECHK")), len(ins))
    return a - before, wait - a


def frame_loop(ins):
    """(first, last) instruction of the longest backward branch (16-byte instructions)"""
    best = (0, 0)
    for i, s in enumerate(ins):
        m = re.match(r"BRA(\.\S+)?\s.*?0x([0-9a-f]+)$", s)
        if m and int(m.group(2), 16) // 16 < i and i - int(m.group(2), 16) // 16 > best[1] - best[0]:
            best = (int(m.group(2), 16) // 16, i)
    return best


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    want = args[1] if len(args) > 1 else "ber_tconv2_kernel"
    for name, ins in kernels(args[0]).items():
        if want not in name:
            continue
        c = counts(ins)
        lo, hi = frame_loop(ins)
        print(f"{name}: {len(ins)} instructions, frame loop {hi - lo + 1}" +
              (f", tx->arrive {c[0]}, arrive->wait {c[1]}" if c else ", no BAR.ARV"))
        if "--opcodes" in sys.argv:
            ops = collections.Counter(i.split()[0].split(".")[0] for i in ins[lo:hi + 1])
            print("    " + " ".join(f"{k} {v}" for k, v in ops.most_common()))
        if "--regions" in sys.argv:
            cuts = [0] + [i for i, s in enumerate(ins) if s.startswith(("BAR.", "SYNCS.PHASECHK"))] + [len(ins)]
            for a, b in zip(cuts, cuts[1:]):
                print(f"    {a:5d} .. {b:5d}  {b - a:4d}  {ins[a][:48]}")


if __name__ == "__main__":
    main()
