#!/usr/bin/env python
"""Writes profiles/<round>_sass_hot_kernels.txt from the built library: per hot kernel the SASS instruction count, the opcode
histogram and a few telling excerpts (kCull's chain-product step, kSortPass' ballot step). CPU only (cuobjdump).

  python tools/sass_summary.py [out.txt]
"""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
LIB = ROOT / "garden_b200" / "libgarden_sceneprep.so"
OUT = Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "profiles" / "r2_sass_hot_kernels.txt"
HOT = ["kPrepassILj5E", "kCompactSurvivorsILb0E", "kCullILj5ELb0E", "kCullILj5ELb1E", "kClassifyILj5E", "kScanChunks", "kScatter",
       "kSortPass", "kEmit", "kTreePartitionILb1E", "kMergeTreeILb1E", "kMergeTreeILb0E", "kPackByDestination", "kSplitRuns",
       "kInstances", "kAnimate"]

sass = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True, check=True).stdout
kernels, name = collections.OrderedDict(), None
for line in sass.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        name = m.group(1)
        kernels[name] = []
    elif name and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
        kernels[name].append(line.rstrip())


def opcode(line):
    t = line.split("*/", 1)[1].strip()
    t = re.sub(r"^@!?U?P\d+\s+", "", t)
    return t.split()[0].rstrip(";")


def excerpt(lines, pred, before=2, count=22):
    for i, l in enumerate(lines):
        if pred(lines, i):
            return [x[:118] for x in lines[max(i - before, 0):i + count]]
    return []


out = ["# SASS of the hot kernels (cuobjdump -sass libgarden_sceneprep.so, sm_100a; written by tools/sass_summary.py): per kernel",
       "# the instruction count, the opcode histogram and a few excerpts. Packed FP32 (FFMA2 / FMUL2) in the chain products and the",
       "# conservative classifier; no UTMALDG / UBLKCP / LDGSTS anywhere: see DESIGN.md 8 (why no bulk-async copies).", ""]
total_bulk = sum(1 for ls in kernels.values() for l in ls if re.search(r"UTMALDG|UBLKCP|LDGSTS|UTMASTG", l))
out.append(f"bulk-async / TMA instructions in the whole library: {total_bulk}")
out.append("")
for want in HOT:
    for name, lines in kernels.items():
        if want not in name:
            continue
        hist = collections.Counter(opcode(l) for l in lines)
        out.append(f"== {name}: {len(lines)} instructions")
        out.append("   " + ", ".join(f"{k} {v}" for k, v in hist.most_common(26)))
        if "kCullILj5ELb0E" in name:
            ex = excerpt(lines, lambda ls, i: all("FFMA2" in x or "FMUL2" in x for x in ls[i:i + 3]), 2, 30)
            out.append("   -- chain-product step (M <- L(parent) * M):")
            out += ["   " + x for x in ex]
        if "kSortPass" in name:
            ex = excerpt(lines, lambda ls, i: "R2P" in ls[i], 1, 26)
            out.append("   -- digit peers of one key: predicates of the 8 digit bits (R2P), then vote / and-not / and per bit:")
            out += ["   " + x for x in ex]
        if "kMergeTreeILb0E" in name:
            ex = excerpt(lines, lambda ls, i: "LDG" in ls[i] and sum("LDG" in x for x in ls[i:i + 30]) >= 12, 0, 34)
            out.append("   -- staging of a tile: all loads of the thread in flight before the first shared store:")
            out += ["   " + x for x in ex]
        out.append("")
        break
OUT.write_text("\n".join(out) + "\n")
print(OUT, len(out), "lines")
