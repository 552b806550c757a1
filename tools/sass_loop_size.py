"""Byte size of kernel C's evaluation loops (all roles) in a SASS dump: python tools/sass_loop_size.py <dump.sass> [function substring]
The loops must fit the SM's ~32 KB instruction cache together (tools/ubench/icache2.cu)."""
import re, sys
fn = sys.argv[2] if len(sys.argv) > 2 else "glg_step_units_kernelIdLb0ELb0ELb0E"
cur, lo, hi, n64 = None, None, None, 0
for line in open(sys.argv[1]):
    if "Function :" in line:
        if cur and fn in cur and lo is not None:
            print(f"{cur}: loops {hex(lo)}..{hex(hi)} = {(hi - lo) / 1024:.1f} KB")
        cur, lo, hi = line.split("Function :")[1].strip(), None, None
        continue
    if cur and fn in cur:
        m = re.match(r"\s*/\*([0-9a-f]+)\*/\s+(.*?);", line)
        if not m:
            continue
        a, t = int(m.group(1), 16), m.group(2)
        if re.search(r"BAR\.(SYNC|ARV)[.A-Z_]* (0x[1-3]|R\d+),", t) or re.search(r"@!?P\d BAR", t):
            lo = a if lo is None else lo
            hi = a
if cur and fn in cur and lo is not None:
    print(f"{cur}: loops {hex(lo)}..{hex(hi)} = {(hi - lo) / 1024:.1f} KB")
