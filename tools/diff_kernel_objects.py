#!/usr/bin/env python
"""Compare two builds of a CUDA object (e.g. kernels.o before and after a refactor), kernel by kernel.

Reports kernels present in only one build, every kernel whose REG / STACK / LOCAL
(`cuobjdump -res-usage`) rose, and every kernel whose `cuobjdump -sass` listing differs, apart from
the kernels named by --changed (regular expressions on the mangled name), whose code is expected to
change.  Kernels are matched by name, so a change in the order of functions in the file does not
count.  Exits 1 on any finding.
usage: diff_kernel_objects.py OLD.o NEW.o [--changed REGEX ...]"""
import argparse
import re
import subprocess
import sys


def cuobjdump(flag, path):
    return subprocess.run(["cuobjdump", flag, path], capture_output=True, text=True, check=True).stdout


def usage(path):
    return {name: tuple(int(v) for v in vals) for name, *vals in re.findall(
        r"Function (\S+):\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", cuobjdump("-res-usage", path))}


def sass(path):
    blocks = re.split(r"\n\s*Function : ", cuobjdump("-sass", path))[1:]
    return {b.split("\n", 1)[0].strip(): b.split("\n", 1)[1] for b in blocks}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--changed", nargs="*", default=[], help="kernels whose SASS may differ")
    a = ap.parse_args()
    u0, u1 = usage(a.old), usage(a.new)
    s0, s1 = sass(a.old), sass(a.new)
    bad = 0
    for name in sorted(set(u0) ^ set(u1)):
        print("only in %s: %s" % (a.old if name in u0 else a.new, name))
        bad += 1
    common = sorted(set(u0) & set(u1))
    for name in common:
        rose = [k for k, v0, v1 in zip(("REG", "STACK", "LOCAL"), u0[name], u1[name]) if v1 > v0]
        if rose:
            print("%s rose: %s -> %s %s" % ("/".join(rose), u0[name], u1[name], name))
            bad += 1
    expected = [re.compile(r) for r in a.changed]
    same = 0
    for name in common:
        if any(r.search(name) for r in expected):
            continue
        if s0.get(name) != s1.get(name):
            print("SASS differs: %s" % name)
            bad += 1
        else:
            same += 1
    print("%d kernels in both builds, %d with identical SASS, %d findings" % (len(common), same, bad))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
