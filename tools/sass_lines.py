#!/usr/bin/env python
"""Static SASS instructions per source line of one kernel, from the line table of a -lineinfo build.

    python tools/sass_lines.py OBJ KERNEL_SUBSTRING [--file fused_blk.cuh] [--lines FIRST-LAST]

OBJ is a host object or shared library with embedded sm_100a code (e.g. csrc/_obj/fused_lpr.o).  Each instruction
is charged to the OUTERMOST frame of its inline chain that lies in --file inside --lines, so that a helper inlined at
a call site (absdiff4 on the straight feature path, blk_round at the round loop) counts at that call site.  Prints
`line  count  source text` for every line that received an instruction; instructions that fall outside the range are
summed as `other`.  Needs cuobjdump / nvdisasm (CUDA toolkit), no GPU.
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ap = argparse.ArgumentParser()
ap.add_argument("obj")
ap.add_argument("kernel", help="substring of the mangled kernel name, e.g. lpr_kernelILb1ELb1ELb0ELb0ELb1ELb0E")
ap.add_argument("--file", default="fused_blk.cuh")
ap.add_argument("--lines", default="1-1000000", help="source line range, e.g. the t loop of blk_stream")
args = ap.parse_args()
lo, hi = (int(x) for x in args.lines.split("-"))

with tempfile.TemporaryDirectory() as tmp:
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(args.obj)], cwd=tmp, check=True, capture_output=True)
    cubins = [f for f in os.listdir(tmp) if f.endswith(".cubin")]
    text = ""
    for c in cubins:
        out = subprocess.run(["nvdisasm", "-gi", "-c", os.path.join(tmp, c)], capture_output=True, text=True, check=True).stdout
        if args.kernel in out:
            text = out
            break
if not text:
    sys.exit(f"kernel {args.kernel!r} not found")

frame_re = re.compile(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?')
ins_re = re.compile(r"/\*[0-9a-f]{4,}\*/\s+(.*?);")
counts = collections.Counter()
other = 0
inside = False
chain = []  # (file, line) innermost first, as nvdisasm prints it
fresh = True
src_path = None
for ln in text.splitlines():
    if ln.startswith("\t.section") or ln.startswith("//----"):
        inside = args.kernel in ln and ".text." in ln
        continue
    if not inside:
        continue
    m = frame_re.search(ln)
    if m:
        if fresh:
            chain = []
            fresh = False
        chain.append((m.group(1), int(m.group(2))))
        continue
    if ins_re.search(ln):
        fresh = True
        hit = None
        for f, l in chain:  # innermost -> outermost: keep the last frame in range
            if os.path.basename(f) == args.file and lo <= l <= hi:
                hit = l
                src_path = f
        if hit is None:
            other += 1
        else:
            counts[hit] += 1

src = open(src_path).read().splitlines() if src_path and os.path.exists(src_path) else []
for l in sorted(counts):
    txt = src[l - 1].strip() if l - 1 < len(src) else ""
    print(f"{l:5d} {counts[l]:5d}  {txt[:110]}")
print(f"total in {args.file}:{lo}-{hi}: {sum(counts.values())}   other: {other}")
