#!/usr/bin/env python
"""Per-kernel counts of the SASS mnemonics that prove which hardware paths a kernel uses (profiles/r03_sass_summary.md).
    python tools/sass_summary.py > profiles/r03_sass_summary.md        (no GPU needed: cuobjdump on the built library)"""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
LIB = ROOT / "audiolm_pytorch_b200" / "libalm_b200.so"
COLS = ["UTCHMMA", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UBLKCP", "LDGSTS", "UTCBAR", "BRA.U.ANY", "HMMA", "FFMA", "FFMA2", "SHFL", "WARPSYNC", "MUFU"]

sass = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True, check=True).stdout
names = subprocess.run(["cu++filt"], input="\n".join(re.findall(r"Function : (\S+)", sass)), capture_output=True, text=True).stdout.split("\n")
counts, order, cur, ni = {}, [], None, 0
for line in sass.split("\n"):
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = names[ni].replace("(int)", "").replace("(bool)", "").split("(")[0].replace("void ", "")
        ni += 1
        if cur not in counts:
            counts[cur] = collections.Counter()
            order.append(cur)
        continue
    m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m and cur:
        op = m.group(1)
        for c in COLS:
            if op == c or op.startswith(c + "."):
                counts[cur][c] += 1
print("# SASS mnemonics per kernel of libalm_b200.so (sm_100a)\n")
print("`python tools/sass_summary.py` (`cuobjdump -sass audiolm_pytorch_b200/libalm_b200.so`, counted per function; __noinline__ device")
print("functions are part of their kernel's function).  UTCHMMA = tcgen05.mma, LDTM / STTM = tcgen05.ld / st, UTMALDG / UTMASTG = TMA")
print("tensor load / store, UBLKCP = cp.async.bulk, LDGSTS = cp.async, UTCBAR = tcgen05.commit, `BRA.U.ANY` = per-instruction ELECT")
print("loops (0 in the MMA / TMA issue paths since the elect-one rewrite), HMMA = mma.sync (none: no legacy tensor-core path), FFMA2 = packed fma.rn.f32x2, WARPSYNC = shuffles the")
print("compiler could not prove converged.\n")
print("| kernel | " + " | ".join(COLS) + " |")
print("|---|" + "---|" * len(COLS))
rows = sorted(order, key=lambda k: (-counts[k]["UTCHMMA"], -counts[k]["UBLKCP"], -counts[k]["LDGSTS"], k))
for k in rows:
    print(f"| `{k}` | " + " | ".join(str(counts[k][c]) for c in COLS) + " |")
