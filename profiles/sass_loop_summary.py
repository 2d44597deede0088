"""Static SASS size of the combinatorial run kernels: per kernel, the instruction count of the whole function and of
its outermost loop (the episode's step loop: the widest backward branch), and the count of a few opcodes inside that
loop.  Static counts, not a measurement: each loop instruction is issued once per warp per step.
usage: python profiles/sass_loop_summary.py [object file] [kernel name filter] > profiles/rNN_sass_loop_summary.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
obj = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "d2d-ppo_b200", "csrc", "build", "env_comb_w4.o")
flt = sys.argv[2] if len(sys.argv) > 2 else "comb_run_kernel"
sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
COLS = ["IMAD.WIDE.U32", "STG", "LDS", "LDC", "BRA", "ISETP", "FSEL", "SEL", "LOP3", "IADD3"]

funcs, cur = collections.OrderedDict(), None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        cur = m.group(1)
        funcs[cur] = []
        continue
    m = re.search(r"/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[T\d]+\s+)?([A-Z0-9_.]+)([^;]*);", line)
    if cur and m:
        funcs[cur].append((int(m.group(1), 16), m.group(2), m.group(3)))

names = dict(zip(funcs, subprocess.run(["c++filt"], input="\n".join(funcs), capture_output=True,
                                       text=True).stdout.splitlines()))
print(f"static SASS of {os.path.basename(obj)}, nvcc 12.9 -gencode arch=compute_100a,code=sm_100a")
print(f"{'kernel':52s} {'total':>6s} {'loop':>6s}" + "".join(f"{c:>14s}" for c in COLS))
for f, ins in funcs.items():
    name = names[f].replace("d2d::", "").replace("void ", "")
    if flt not in name:
        continue
    lo, hi = None, None
    for addr, op, args in ins:            # the widest backward branch spans the outer loop
        if op.startswith("BRA"):
            t = re.search(r"0x([0-9a-f]+)", args)
            if t and int(t.group(1), 16) < addr and (lo is None or addr - int(t.group(1), 16) > hi - lo):
                lo, hi = int(t.group(1), 16), addr
    body = [op for addr, op, _ in ins if lo is not None and lo <= addr <= hi]
    cnt = collections.Counter()
    for op in body:
        for c in COLS:
            if op == c or op.startswith(c + "."):
                cnt[c] += 1
    print(f"{name[:52]:52s} {len(ins):6d} {len(body):6d}" + "".join(f"{cnt[c]:14d}" for c in COLS))
