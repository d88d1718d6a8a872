"""Compares the SASS of the kernels two object files have in common, instruction for instruction (cuobjdump -sass).

    python tools/sass_compare.py old/trace_kernels.o new/trace_kernels.o [--match traceKernel]

Prints, per kernel whose name contains --match, whether its instruction list is the same, and the kernels only one side has; exit code 1
when a matched kernel differs.  A change that shares device code between kernels (e.g. the base-colour tap of the trace and guide-buffer
kernels) shows with it that the trace kernels' machine code did not move."""
import argparse
import re
import subprocess
import sys


def kernels(obj):
    out, cur = {}, None
    text = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s*(.*?)\s*;", line)
        if m and cur is not None:
            cur.append(m.group(1))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--match", default="traceKernel")
    ap.add_argument("--rename", action="append", default=[], metavar="NEW=OLD",
                    help="replace NEW by OLD in the new object's kernel names, e.g. when a template parameter with a default was added")
    a = ap.parse_args()
    old, new = kernels(a.old), kernels(a.new)
    for r in a.rename:
        frm, to = r.split("=", 1)
        new = {k.replace(frm, to): v for k, v in new.items()}
    names = sorted(k for k in old if a.match in k and k in new)
    diff = [k for k in names if old[k] != new[k]]
    for k in names:
        print(("differs  " if k in diff else "same     ") + f"{len(old[k]):6d} -> {len(new[k]):6d}  {k}")
    print(f"{len(names) - len(diff)} of {len(names)} matched kernels identical ({sum(len(old[k]) for k in names)} instructions); "
          f"only in old: {sorted(set(old) - set(new))}; only in new: {sorted(set(new) - set(old))}")
    sys.exit(1 if diff else 0)


if __name__ == "__main__":
    main()
