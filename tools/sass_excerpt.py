"""profiles/r2_sass_hot_loop.txt: SASS evidence for the headline kernel from `cuobjdump -sass libglgym.so`:
  * the TMA staging of the weather tile in the prologue (UBLKCP / SYNCS lines with their addresses),
  * address range and byte size of every role loop (group warps + owners) and of all of them together,
  * local-memory instructions (LDL / STL: register spills, per-thread arrays) inside vs outside the loops,
  * the owner loop and the shortest group loop in full.
usage: python tools/sass_excerpt.py [libglgym.so] [function substring] > profiles/r2_sass_hot_loop.txt"""
import os, re, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools", "sasssim"))
from parse import functions, parse  # noqa: E402
import sim2  # noqa: E402

lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "greenlight-gym2_b200", "glgym", "libglgym.so")
fn = sys.argv[2] if len(sys.argv) > 2 else "glg_step_units_kernelIdLb0ELb0ELb0E"
dump = "/tmp/_sass_excerpt.sass"
open(dump, "w").write(subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout)
arch = re.search(r"arch = (sm_\w+)", open(dump).read())
print(f"# {os.path.basename(lib)}: {arch.group(1) if arch else '?'}; kernel {fn} (fp64, nominal parameter structure, latency layout)")
for name, lines in functions(dump):
    if fn not in name:
        continue
    ins = parse(lines)
    print(f"# {name}: {len(ins)} instructions, {(ins[-1].addr + 16) / 1024:.1f} KB")
    print("\n## TMA weather staging (prologue): cp.async.bulk + mbarrier")
    for x in ins:
        if x.op.startswith(("UBLKCP", "SYNCS")):
            print(f"  {x.addr:#07x}  {x.text[:110]}")
    loops = sim2.loops_of(ins)
    in_loop = set()
    print("\n## role loops (one per group role, the surface role shared by three warps, one owner loop shared by four)")
    for kind, a, b in loops:
        body = ins[a:b + 1]
        nl = sum(1 for x in body if x.op.startswith(("LDL", "STL")))
        n64 = sum(1 for x in body if x.op.startswith(("DFMA", "DMUL", "DADD", "DSETP", "MUFU.RCP64H", "MUFU.RSQ64H")))
        in_loop.update(range(a, b + 1))
        print(f"  {kind:5s} {ins[a].addr:#07x}..{ins[b].addr:#07x}  {len(body):4d} instr  {len(body) * 16:5d} B  FP64 {n64:3d}  LDL/STL {nl}")
    lo, hi = min(a for _, a, _ in loops), max(b for _, _, b in loops)
    print(f"  all loops span {ins[lo].addr:#07x}..{ins[hi].addr:#07x} = {(ins[hi].addr - ins[lo].addr + 16) / 1024:.1f} KB "
          f"(instruction cache ~32 KB, tools/ubench/icache2.cu)")
    loc = [(k, x) for k, x in enumerate(ins) if x.op.startswith(("LDL", "STL"))]
    print(f"\n## local memory: {len(loc)} LDL/STL instructions in the kernel, {sum(1 for k, _ in loc if k in in_loop)} of them inside a role loop")
    for k, x in loc[:12]:
        print(f"  {x.addr:#07x}  {'LOOP ' if k in in_loop else 'outside'}  {x.text[:100]}")
    if len(loc) > 12:
        print(f"  ... ({len(loc) - 12} more, all {'outside the loops' if not any(k in in_loop for k, _ in loc) else 'see above'})")
    for title, pick in (("owner loop", [l for l in loops if l[0] == "owner"][0]),
                        ("shortest group loop", min((l for l in loops if l[0] == "group"), key=lambda l: l[2] - l[1]))):
        _, a, b = pick
        print(f"\n## {title} {ins[a].addr:#07x}..{ins[b].addr:#07x}")
        for x in ins[a:b + 1]:
            print(f"  {x.addr:#07x}  {x.text[:120]}")
