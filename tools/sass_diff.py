"""Compare the SASS of two builds function by function.

    python tools/sass_diff.py OLD_OBJ_DIR NEW_OBJ_DIR

Runs `cuobjdump -sass` on every object file (*.o) of both directories, splits each listing at its `Function :` headers
and compares each function's instructions and encodings.  Prints one line per object and a line for every function
that differs or exists on one side only; a function that exists on one side only but has the same SASS as a function
that exists on the other side only is reported as renamed.  Anonymous-namespace ids (`_GLOBAL__N__<hash>`, which
depend on where the source was compiled) are blanked in the names.  Exits with 1 if anything differs, renames included.
"""
import argparse
import os
import re
import subprocess
import sys


def functions(obj):
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = re.sub(r"_GLOBAL__N__[0-9a-f]+", "_GLOBAL__N__", m.group(1))
            funcs[name] = []
        elif name is not None and line.strip() and not line.lstrip().startswith(("....", ".section", "Fatbin", "code for")):
            funcs[name].append(line.strip())
    return {k: "\n".join(v) for k, v in funcs.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("old")
    ap.add_argument("new")
    a = ap.parse_args()
    names = sorted(set(f for d in (a.old, a.new) for f in os.listdir(d) if f.endswith(".o")))
    differ = False
    for obj in names:
        po, pn = os.path.join(a.old, obj), os.path.join(a.new, obj)
        if not os.path.exists(po) or not os.path.exists(pn):
            print(f"{obj}: only in {'new' if os.path.exists(pn) else 'old'}")
            differ = True
            continue
        fo, fn = functions(po), functions(pn)
        same = [k for k in fo if k in fn and fo[k] == fn[k]]
        changed = [k for k in fo if k in fn and fo[k] != fn[k]]
        gone = [k for k in fo if k not in fn]
        added = [k for k in fn if k not in fo]
        print(f"{obj}: {len(same)} identical, {len(changed)} changed, {len(gone)} only in old, {len(added)} only in new")
        for k in changed:
            print(f"  changed: {k}")
        for k in gone:
            to = [n for n in added if fn[n] == fo[k]]
            if to:
                added.remove(to[0])
                print(f"  renamed, same SASS: {k} -> {to[0]}")
            else:
                print(f"  only in old: {k}")
        for k in added:
            print(f"  only in new: {k}")
        differ |= bool(changed or gone or added)
    sys.exit(1 if differ else 0)


if __name__ == "__main__":
    main()
