#!/usr/bin/env python
"""Register / spill figures of ONE kernel of a .cu file without building the library (nvcc -ptx, cut the entry out, ptxas -v):
    tools/kernel_regs.py wavefront.cu k_shadeILb0ELb0ELb0E [-DFLAG ...] [--maxrregcount N]
The .maxntid / .minnctapersm directives of the entry (its __launch_bounds__) are honoured unless --maxrregcount is given."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "path-tracing_b200", "csrc")
src, want = sys.argv[1], sys.argv[2]
rest = sys.argv[3:]
maxr = None
if "--maxrregcount" in rest:
    i = rest.index("--maxrregcount")
    maxr = rest[i + 1]
    del rest[i:i + 2]
out = os.path.join(ROOT, "scratch")
os.makedirs(out, exist_ok=True)
ptx = os.path.join(out, "kr.ptx")
subprocess.check_call(["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=compute_100a", "-lineinfo", "-fmad=false",
                       "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-ptx", src, "-o", ptx] + rest, cwd=CSRC)
text = open(ptx).read()
# split into top-level items; keep everything that is not an entry, plus the wanted entry
parts = re.split(r"(?m)^(?=\.(?:visible |weak )?\.?entry )", text)
keep = [parts[0]]
found = 0
for p in parts[1:]:
    # an entry runs to its closing brace at column 0; what follows (globals, functions) is kept
    depth, pos, started = 0, 0, False
    for line in p.splitlines(keepends=True):  # the entry ends where its braces balance (inline asm nests more)
        code = line.split("//")[0]
        depth += code.count("{") - code.count("}")
        started = started or "{" in code
        pos += len(line)
        if started and depth == 0:
            break
    body, tail = p[:pos], p[pos:]
    name = re.match(r"\.(?:visible |weak )?\.?entry (\S+?)\(", body)
    if name and want in name[1]:
        if maxr:
            body = re.sub(r"\.minnctapersm \d+\n?", "", body)
        keep.append(body)
        found += 1
    keep.append(tail)
if not found:
    sys.exit(f"no entry matching {want}")
cut = os.path.join(out, "kr_cut.ptx")
open(cut, "w").write("".join(keep))
cmd = ["ptxas", "-arch=sm_100a", "-v", "-O3", cut, "-o", os.path.join(out, "kr.cubin")]
if maxr:
    cmd += ["-maxrregcount", maxr]
r = subprocess.run(cmd, capture_output=True, text=True)
for l in r.stderr.splitlines():
    if "registers" in l or "spill" in l or "error" in l.lower():
        print(l.strip())
