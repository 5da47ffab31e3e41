#!/usr/bin/env python3
"""Compare the SASS of the kernels in two builds of the library, kernel by kernel.

    python tools/sass_diff.py OLD_BUILD_DIR NEW_BUILD_DIR [OBJ ...] [--map OLD=NEW ...]

OBJ names object files in both directories (default: chain_rx_t4.o and every sweep*.o of the new build).  Kernels are
matched by demangled name without the parameter list; --map renames a kernel of the old build (for example a template that
gained a parameter: --map 't4_post_kernel<(bool)1, (bool)0>=t4_post_kernel<(bool)1, (bool)0, (bool)0>').  The address column and the
/* ... */ encodings are stripped, so two kernels compare equal when their instruction sequences are equal.  Prints one line
per kernel (identical / DIFFERENT with the count of differing lines and both instruction counts / only in one build) and
exits 1 when any matched kernel differs.  Needs cuobjdump and cu++filt from the CUDA toolkit, no GPU.
"""
import argparse
import difflib
import glob
import os
import re
import subprocess
import sys


def kernels(obj):
    """{demangled name without parameters: [instruction lines]} of one object file."""
    out = subprocess.run(["cuobjdump", "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*(/\*.*\*/)?\s*$", line)
        if name and m and m.group(1):
            funcs[name].append(m.group(1).rstrip(" ;"))
    if not funcs:
        return {}
    names = list(funcs)
    dem = subprocess.run(["cu++filt"], input="\n".join(names), check=True, capture_output=True, text=True).stdout.splitlines()
    res = {}
    for mangled, d in zip(names, dem):
        d = re.sub(r"^void ", "", d)
        depth, cut = 0, len(d)
        for i, c in enumerate(d):                       # drop the parameter list: the first '(' outside template brackets
            if c == "<":
                depth += 1
            elif c == ">":
                depth -= 1
            elif c == "(" and depth == 0:
                cut = i
                break
        res[d[:cut]] = funcs[mangled]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("objs", nargs="*")
    ap.add_argument("--map", action="append", default=[], help="OLD=NEW kernel rename")
    a = ap.parse_args()
    rename = dict(m.split("=", 1) for m in a.map)
    objs = a.objs or ["chain_rx_t4.o"] + sorted(os.path.basename(p) for p in glob.glob(os.path.join(a.new, "sweep*.o")))
    differ = False
    for obj in objs:
        old = {rename.get(k, k): v for k, v in kernels(os.path.join(a.old, obj)).items()}
        new = kernels(os.path.join(a.new, obj))
        print(f"== {obj}")
        for k in sorted(set(old) | set(new)):
            if k not in new:
                print(f"  only in old   {k}")
            elif k not in old:
                print(f"  only in new   {k} ({len(new[k])} instructions)")
            elif old[k] == new[k]:
                print(f"  identical     {k} ({len(new[k])} instructions)")
            else:
                differ = True
                n = sum(1 for l in difflib.unified_diff(old[k], new[k], n=0, lineterm="") if l[:1] in "+-" and l[:3] not in ("+++", "---"))
                print(f"  DIFFERENT     {k} ({n} differing lines; {len(old[k])} -> {len(new[k])} instructions)")
    return 1 if differ else 0


if __name__ == "__main__":
    sys.exit(main())
