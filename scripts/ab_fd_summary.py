#!/usr/bin/env python
"""Medians and spreads of an A/B written by scripts/ab_fd_transforms.sh (time mode), and the per-call-site live times of its
two CMF_TRACE=1 runs (a call site is the function and line of the post_launch() after a launch).
    python scripts/ab_fd_summary.py OUT_DIR"""
import glob
import json
import os
import re
import statistics
import sys


def last_json(path):
    lines = [l for l in open(path) if l.startswith("{")]
    return json.loads(lines[-1]) if lines else None


def main():
    out = sys.argv[1]
    print(open(os.path.join(out, "gpu.txt")).read().strip())
    for key in ("ms_per_step", "value_direct_loss", "value_calibrated_loss"):
        row = []
        for side in "AB":
            vals = []
            for p in sorted(glob.glob(os.path.join(out, f"time_{side}_*.json"))):
                d = last_json(p)
                if d is None:
                    continue
                v = d[key]
                vals.append(v["value"] if isinstance(v, dict) else v)
            if vals:
                row.append(f"{side}: median {statistics.median(vals):.3f} [{min(vals):.3f}, {max(vals):.3f}] n={len(vals)}")
        print(f"{key:24s}", "   ".join(row))
    # CMF_TRACE lines: "CMF_TRACE <fn>:<line> n=<count> total <ms> ms  mean <ms> ms  <pct>%"
    for side in "AB":
        p = os.path.join(out, f"trace_{side}.err")
        if not os.path.exists(p):
            continue
        rows = []
        for line in open(p):
            m = re.match(r"CMF_TRACE (\S+)\s*:(\d+)\s+n=(\d+)\s+total\s+([\d.]+) ms\s+mean\s+([\d.]+) ms", line)
            if m:
                rows.append((m.group(1), int(m.group(2)), int(m.group(3)), float(m.group(4)), float(m.group(5))))
        print(f"trace {side}:")
        for r in sorted(rows, key=lambda r: -r[3]):
            print(f"   {r[0]:28s}:{r[1]:<5d} n={r[2]:<6d} total {r[3]:10.3f} ms  mean {r[4]:8.4f} ms")


if __name__ == "__main__":
    main()
