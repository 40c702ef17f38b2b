"""Join an `ncu --page source --csv` SASS dump with `nvdisasm -g -c` line info to rank source
lines by executed warp instructions.  Usage: sass_lines.py ncu_sass.csv nvdisasm.txt kernel_substring"""
import collections
import csv
import os
import re
import sys

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rmi_b200", "csrc")
ncu_csv, dis_txt, kname = sys.argv[1:4]
rows = list(csv.reader(open(ncu_csv)))
hi = next(i for i, r in enumerate(rows) if "Source" in r and "Instructions Executed" in r)
hdr = rows[hi]
iS, iE, iSm = hdr.index("Source"), hdr.index("Instructions Executed"), hdr.index("# Samples")
insts = [(r[iS].strip(), int(r[iE]), int(r[iSm]) if r[iSm].isdigit() else 0) for r in rows[hi + 1:]
         if len(r) > iE and r[iE].isdigit()]

# walk nvdisasm output: find the function, collect (line, opcode) per instruction in order
lines = open(dis_txt, errors="replace").read().split("\n")
start = next(i for i, l in enumerate(lines) if l.startswith("\t.text.") is False and re.match(r"\s*\.text\..*" + re.escape(kname), l))
cur = None
seq = []
inline_stack = ""
for l in lines[start + 1:]:
    if re.match(r"\s*\.text\.", l) or l.startswith("//--------------------- .text"):
        if seq:
            break
    m = re.search(r'//## File "([^"]+)", line (\d+)(.*)', l)
    if m:
        cur = (m.group(1).split("/")[-1], int(m.group(2)), m.group(3).strip())
        continue
    m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(.+?);", l)
    if m:
        seq.append((cur, m.group(1).strip()))
print("ncu instructions", len(insts), "nvdisasm instructions", len(seq))
agg = collections.Counter()
samp = collections.Counter()
n = min(len(insts), len(seq))
tot = 0
for (src, e, s), (loc, op) in zip(insts[:n], seq[:n]):
    key = (loc[0], loc[1]) if loc else ("?", 0)
    agg[key] += e
    samp[key] += s
    tot += e
srcs = {}
for (f, ln), c in agg.most_common(40):
    if f not in srcs:
        try:
            srcs[f] = open(os.path.join(CSRC, f)).read().split("\n")
        except Exception:
            srcs[f] = []
    text = srcs[f][ln - 1].strip()[:100] if 0 < ln <= len(srcs[f]) else ""
    print(f"{100 * c / tot:5.1f}% {c:11d} samp {samp[(f, ln)]:6d}  {f}:{ln}  {text}")
