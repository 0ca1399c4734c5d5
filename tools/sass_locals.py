"""Local-memory traffic (LDL / STL) of one kernel: per barrier-delimited region (numbered as tools/sass_regions.py
numbers them), each access with its source line and stack offset, then per stack slot the source lines that write
and read it.
usage: nvcc ... -lineinfo -cubin -o k.cubin unit.cu; nvdisasm --print-line-info k.cubin |
       python tools/sass_locals.py kernel-substring [region ...]"""
import re, sys, collections
pat = sys.argv[1]
want = set(int(x) for x in sys.argv[2:])
on = False
src = "?"
region = 0
recs = []  # (region, op, off, srcline, addr)
for l in sys.stdin:
    if l.startswith("//---------------------") and ".text." in l:
        on = pat in l
        region = 0
        continue
    if not on:
        continue
    m = re.search(r'//## File "([^"]+)", line (\d+)', l)
    if m:
        src = f"{m.group(1).split('/')[-1]}:{m.group(2)}"
        continue
    m = re.search(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_.]+)(.*)", l)
    if not m:
        continue
    op = m.group(3)
    if op.startswith("LDL") or op.startswith("STL"):
        o = re.search(r"\[R1(\+0x([0-9a-f]+))?\]", m.group(4))
        off = int(o.group(2), 16) if o and o.group(2) else 0
        recs.append((region, op, off, src, m.group(1)))
    if op.startswith("BAR") or op.startswith("WARPSYNC"):
        region += 1
for r in sorted(set(x[0] for x in recs)):
    if want and r not in want:
        continue
    rr = [x for x in recs if x[0] == r]
    print(f"region {r}: {sum(1 for x in rr if x[1].startswith('LDL'))} LDL, {sum(1 for x in rr if x[1].startswith('STL'))} STL")
    for x in rr:
        print(f"   {x[4]} {x[1]:10s} [0x{x[2]:03x}]  {x[3]}")
print("slots: offset -> written at / read at")
slots = collections.defaultdict(lambda: (set(), set()))
for x in recs:
    slots[x[2]][0 if x[1].startswith("STL") else 1].add(x[3].split(":")[-1])
for off in sorted(slots):
    w, rd = slots[off]
    print(f"  0x{off:03x}: W {sorted(w, key=int)}  R {sorted(rd, key=int)}")
