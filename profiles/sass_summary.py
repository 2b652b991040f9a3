#!/usr/bin/env python
"""Opcode histogram of the shipped kernels (cuobjdump -sass of the built libbmx.so): the proof, kept in the
repository, that the bulk-copy (TMA) path, the mbarrier pipeline, 16-byte shared loads and the warp reductions
are what ships (the .so itself is git-ignored).
    python profiles/sass_summary.py > profiles/sass_r02.txt"""
from __future__ import annotations

import re
import subprocess
import sys
from collections import Counter
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
so = ROOT / "parallel_implementation_of_string_matching_algorithms_opencl_b200" / "libbmx.so"
out = subprocess.run(["cuobjdump", "-sass", str(so)], capture_output=True, text=True, check=True).stdout
WATCH = ["UBLKCP", "SYNCS", "LDS.128", "LDS", "REDUX", "VOTE", "SHFL", "IMAD", "ISETP", "SHF", "LOP3", "ATOMG", "ATOM", "RED", "STG", "LDG",
         "MEMBAR", "FENCE", "ERRBAR", "BAR", "CCTL", "STS", "UTMA", "NANOSLEEP", "LD.E", "ST.E"]
kernels = {}
name = None
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        name = m.group(1)
        kernels[name] = Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m and name:
        kernels[name][m.group(1)] += 1

want = sys.argv[1:] or ["scan_kernelILNS_6FilterE1ELi32768ELb1E", "scan_kernelILNS_6FilterE1ELi32768ELb0E",
                        "scan_kernelILNS_6FilterE2ELi32768ELb1E", "scan_kernelILNS_6FilterE8ELi16384ELb1E", "expand_kernel",
                        "xchg_post_kernel", "xchg_collect_kernel", "multi_split_kernel"]
print(f"# cuobjdump -sass {so.name}: instruction counts per kernel (static), grouped by opcode family")
print("# scan_kernel<Filter, TILE, POSITIONS> (enum Filter, csrc/bmx_internal.h): FilterE1 = kQgram, FilterE2 = kWindow4, "
      "FilterE8 = kMulti; Lb1/Lb0 = positions / count-only")
for k, c in kernels.items():
    if not any(w in k for w in want):
        continue
    total = sum(c.values())
    print(f"\n== {k}  ({total} instructions)")
    fam = Counter()
    for op, n in c.items():
        for w in WATCH:
            if op.startswith(w):
                fam[w if w != "LDS" or not op.startswith("LDS.128") else "LDS.128"] += n
                break
    # exact spellings that matter as evidence
    for op in sorted(c):
        if any(op.startswith(p) for p in ("UBLKCP", "SYNCS", "LDS.128", "REDUX", "VOTE", "ATOMG", "RED", "MEMBAR", "ERRBAR", "NANOSLEEP", "LD.E.STRONG", "ST.E.STRONG", "CCTL")):
            print(f"   {op:42s} {c[op]:5d}")
    print("   families: " + "  ".join(f"{w}={fam[w]}" for w in WATCH if fam[w]))
