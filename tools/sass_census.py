#!/usr/bin/env python
"""SASS census of the SHIPPED library: per kernel, how many of the instructions that prove what the
code runs on (packed FP32 math, bulk-TMA copies, mbarriers, tensor-core / tensor-memory ops,
shuffles).  __graft_entry__.build() writes build/sass_census.txt from the .so it just built, so that
file never describes a stale kernel; run this tool by hand to refresh the committed snapshot
profiles/sass_census.txt with a kernel change.   usage: tools/sass_census.py [lib.so] [out.txt]"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MNEMONICS = ("FFMA2", "FADD2", "FMUL2", "FFMA", "MUFU", "UBLKCP", "UTMALDG", "SYNCS", "SHFL", "UTCHMMA", "UTCQMMA",
             "UTCBAR", "LDTM", "STTM", "UTCCP", "HMMA", "LDGSTS", "DFMA", "STG", "LDG", "LDS", "STS", "BAR")


def census(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    counts = collections.OrderedDict()
    kernel = None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            kernel = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip() or m.group(1)
            kernel = re.sub(r"\(.*", "", kernel)
            counts[kernel] = collections.Counter()
            continue
        m = re.search(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
        if m and kernel:
            op = m.group(1)
            counts[kernel]["_all"] += 1
            if op in MNEMONICS:
                counts[kernel][op] += 1
    return counts


def main(lib=None, dst=None):
    lib = lib or os.path.join(ROOT, "f2cnn_b200", "libf2cnn_b200.so")
    dst = dst or os.path.join(ROOT, "profiles", "sass_census.txt")
    rows = ["# cuobjdump -sass %s: instruction counts per kernel (tools/sass_census.py)" %
            os.path.relpath(lib, ROOT), "# kernel | total | " + " ".join(MNEMONICS)]
    for kernel, c in census(lib).items():
        rows.append("%s | %d | %s" % (kernel, c["_all"], " ".join("%s=%d" % (m, c[m]) for m in MNEMONICS if c[m])))
    with open(dst, "w") as f:
        f.write("\n".join(rows) + "\n")
    return dst


if __name__ == "__main__":
    print(main(*sys.argv[1:3]))
