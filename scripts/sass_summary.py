#!/usr/bin/env python
"""Per-kernel SASS evidence for profiles/: counts of the Blackwell-native mnemonics (B200_PROFILING.md, "What proves a
Blackwell-native kernel") in the in-tree libcmf_sm100.so.   python scripts/sass_summary.py > profiles/r2_sass_summary.md
    python scripts/sass_summary.py [--so PATH] [--match SUBSTRING]   (another build; only kernels whose name contains SUBSTRING)"""
import argparse
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "cmf.jl_b200", "libcmf_sm100.so")
OPS = ["UTCHMMA", "UTMALDG", "LDTM", "UTCBAR", "FFMA2", "FFMA", "FADD2", "FADD", "FMUL2", "FMUL", "DFMA", "LDGSTS", "HMMA", "ATOM",
       "RED", "LDL", "STL"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--so", default=SO)
    ap.add_argument("--match", default="")
    args = ap.parse_args()
    out = subprocess.run(["cuobjdump", "-sass", args.so], capture_output=True, text=True, check=True).stdout
    arch = sorted(set(re.findall(r"arch = (sm_\w+)", out)))
    kern, counts, total = None, collections.OrderedDict(), {}
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kern = m.group(1)
            counts[kern] = collections.Counter()
            total[kern] = 0
            continue
        m = re.search(r"/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and kern:
            op = m.group(1)
            total[kern] += 1
            for o in OPS:
                if op == o or op.startswith(o + "."):
                    counts[kern][o] += 1
                    break
    demangled = subprocess.run(["c++filt"], input="\n".join(counts), capture_output=True, text=True).stdout.splitlines()
    print(f"# SASS summary of {os.path.relpath(args.so, ROOT)} (cuobjdump -sass), architectures:", ", ".join(arch))
    print()
    print("`UTCHMMA` = tcgen05.mma (kind::f16), `UTMALDG` = TMA tensor loads, `LDTM` = tcgen05.ld (TMEM -> registers), `FFMA2` = packed")
    print("fp32x2 FMA (sm_100: the full-rate fp32 path; FADD2 / FMUL2 likewise), `LDL` / `STL` = local-memory (spill) loads / stores, `LDGSTS` = cp.async, `DFMA` = fp64 FMA (the 1e-9 parity path).  No `HMMA`")
    print("(legacy mma.sync) and no floating-point atomics anywhere.")
    print()
    print("| kernel | instructions | " + " | ".join(OPS) + " |")
    print("|---|---:|" + "---:|" * len(OPS))
    tot, shown = collections.Counter(), 0
    for (k, c), name in zip(counts.items(), demangled):
        name = re.sub(r"\(.*", "", name)
        if (total[k] < 40 and not any(c.values())) or args.match not in name:
            continue
        print(f"| `{name}` | {total[k]} | " + " | ".join(str(c[o]) if c[o] else "" for o in OPS) + " |")
        tot.update(c)
        shown += total[k]
    print("| **all kernels** | " + str(shown) + " | " + " | ".join(str(tot[o]) for o in OPS) + " |")


if __name__ == "__main__":
    main()
