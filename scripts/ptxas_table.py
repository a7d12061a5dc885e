#!/usr/bin/env python
"""Registers / spills / shared memory per kernel (ptxas -v) and the Blackwell/Hopper-class SASS mnemonics each kernel
contains (warp REDUX, MATCH, 64-bit shared atomics; cluster barriers UCGABAR_* would show up here).
usage: python scripts/ptxas_table.py > profiles/r02_ptxas_sass_<version>.txt   (no GPU needed: nvcc cross-compiles)"""
import os, re, subprocess, sys, collections
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from urban_road_filter_b200 import build
src = os.path.join(build.CSRC, "urf_api.cu")
out = subprocess.run([build._nvcc(), *build.NVCC_FLAGS, "-Xptxas=-v", "-c", src, "-o", "/tmp/urf_api_ptxas.o"], capture_output=True, text=True).stderr
rows = []
for m in re.finditer(r"Compiling entry function '(\S+)' for 'sm_100a'\n.*?\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers(?:, used (\d+) barriers)?(?:, (\d+) bytes cumulative stack size)?(?:, (\d+) bytes smem)?", out):
    name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip().split("(")[0].replace("urf::", "")
    rows.append((name, int(m.group(5)), int(m.group(2)), int(m.group(3)), int(m.group(4)), int(m.group(8) or 0)))
sass = subprocess.run(["cuobjdump", "-sass", build.LIB], capture_output=True, text=True).stdout
per = collections.defaultdict(collections.Counter)
cur = None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip().split("(")[0].replace("urf::", "")
        continue
    m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m and cur:
        op = m.group(1)
        for tag in ("UCGABAR_ARV", "UCGABAR_WAIT", "REDUX", "MATCH", "ATOMS", "ATOM", "RED", "SHFL", "DSQRT", "MUFU.RSQ64H", "DFMA", "DMUL", "DADD", "LDL", "STL", "BAR.SYNC", "VOTE"):
            if op.startswith(tag):
                per[cur][tag] += 1
                break
        per[cur]["total"] += 1
print("liburf_b200.so built with:", " ".join(build.NVCC_FLAGS))
print(f"{'kernel':28s} {'regs':>4s} {'stack':>5s} {'spill_st':>8s} {'spill_ld':>8s} {'smem_B':>7s} {'sass':>6s}  notable SASS (static counts)")
for name, regs, stack, sst, sld, smem in sorted(rows):
    c = per.get(name, {})
    notes = ", ".join(f"{k} {v}" for k, v in sorted(c.items()) if k != "total" and k not in ("DFMA", "DMUL", "DADD") and v)
    print(f"{name:28s} {regs:4d} {stack:5d} {sst:8d} {sld:8d} {smem:7d} {c.get('total', 0):6d}  {notes}")
print("\nREDUX = warp-wide integer reduce; MATCH = __match_any_sync. No tensor-core or TMA instructions: the path has no dense")
print("contraction and no bulk tile to stage.")
