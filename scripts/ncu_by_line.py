"""Executed warp instructions of lnl_kernel by source line and opcode class.

    python scripts/ncu_by_line.py <report.ncu-rep> <library.so> [launch-id]

Joins the per-instruction counts of an `ncu --set full --import-source on` capture (SASS view)
with the line table of the same binary (nvdisasm -g on the cubin inside the .so): the SASS
instruction order is the same in both.  Prints, per source line (file:line of the innermost
inlined frame), the executed instructions split into FP64-pipe and other, and the opcodes.
"""
import collections
import csv
import io
import os
import re
import subprocess
import sys
import tempfile

rep, so = sys.argv[1], sys.argv[2]
launch = int(sys.argv[3]) if len(sys.argv) > 3 else 0
KERNEL = "lnl_kernel"

tmp = tempfile.mkdtemp()
subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(so)], cwd=tmp, check=True,
               stdout=subprocess.DEVNULL)
cubin = [f for f in os.listdir(tmp) if f.endswith(".cubin")][0]
dis = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cubin)], capture_output=True,
                     text=True).stdout
lines, cur, inside = [], ("?", 0), False
for ln in dis.splitlines():
    if ln.startswith("//---") and ".text." in ln:
        # the production instantiation lnl_kernel<false, false> (no work counters, one cadence)
        inside = KERNEL + "ILb0ELb0EE" in ln
        continue
    if not inside:
        continue
    m = re.search(r'//## File "([^"]+)", line (\d+)', ln)
    if m:
        cur = (os.path.basename(m.group(1)), int(m.group(2)))
        continue
    m = re.match(r'\s+/\*([0-9a-f]{4,})\*/\s+(.*?);', ln)
    if m:
        lines.append((cur, m.group(2).strip()))

sass = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "sass"],
                      capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(sass)))
# kernels are separated by "Kernel Name" rows
blocks, cur_block = [], None
for r in rows:
    if r and r[0] == "Kernel Name":
        cur_block = []
        blocks.append(cur_block)
    elif cur_block is not None:
        cur_block.append(r)
blk = blocks[launch]
hdr = blk[0]
ia, isrc, ith = hdr.index("Instructions Executed"), hdr.index("Source"), hdr.index("Thread Instructions Executed")
inst = [(r[isrc].strip(), int(r[ia]), int(r[ith])) for r in blk[1:] if len(r) > ia and r[ia].isdigit()]
assert len(inst) == len(lines), (len(inst), len(lines))

FP64 = ("DFMA", "DMUL", "DADD", "DSETP", "DMNMX")
by_line = collections.defaultdict(lambda: [0, 0, 0, collections.Counter()])
tot = tot64 = 0
for ((fl, op_dis), (src, n, nth)) in zip(lines, inst):
    s = re.sub(r'^@!?U?P\d+\s+', '', src)
    op = (s.split()[0].rstrip(';') if s else '?').split('.')[0]
    e = by_line[fl]
    e[0] += n
    e[2] += nth
    if op in FP64:
        e[1] += n
        tot64 += n
    e[3][op] += n
    tot += n
print("total executed warp instructions %d, FP64-pipe %.1f%%" % (tot, 100.0 * tot64 / tot))
print("%-28s %7s %7s %7s %6s  %s" % ("file:line", "all%", "fp64%", "other%", "lanes", "top opcodes"))
for fl, e in sorted(by_line.items(), key=lambda kv: -kv[1][0])[:70]:
    ops = " ".join("%s:%.2f" % (o, 100.0 * c / tot) for o, c in e[3].most_common(6))
    print("%-28s %7.2f %7.2f %7.2f %6.1f  %s" % ("%s:%d" % fl, 100.0 * e[0] / tot, 100.0 * e[1] / tot,
                                                 100.0 * (e[0] - e[1]) / tot, e[2] / max(e[0], 1), ops))
