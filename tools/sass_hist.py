"""Opcode histogram per kernel of a cubin/object file.

  python tools/sass_hist.py file.o [name-substring] [--full] [--bodies]

Each line gives the instruction count and the issue slots of DESIGN.md section 4's model (DFMA / DADD / DMUL 2, IMAD.WIDE
2.5, everything else 1).  --full keeps the opcode modifiers (IMAD.WIDE.U32, IMAD.MOV.U32, ...) instead of the bare opcode.
--bodies splits each kernel by loop body: every innermost loop (a backward branch whose range holds no other backward
branch) is listed on its own, the rest of the kernel (loads, absorb, stores, the outer loops' control) as "glue".  In the hash kernels the two largest innermost loops are
Poseidon's full-round body and fused partial-pair body (`#pragma unroll 1` in csrc/poseidon.cuh); the one with more wide
multiplies (twelve S-boxes against two) is the full round."""
import collections
import re
import subprocess
import sys

args = [a for a in sys.argv[1:] if not a.startswith("--")]
full = "--full" in sys.argv
bodies = "--bodies" in sys.argv
out = subprocess.run(["cuobjdump", "-sass", args[0]], capture_output=True, text=True).stdout
pat = args[1] if len(args) > 1 else ""

kernels = collections.OrderedDict()  # name -> [(address, opcode, line)]
name = None
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        name = m.group(1)
        kernels[name] = []
        continue
    m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P[T\d]+\s+)?([A-Z0-9_.]+)(.*)", line)
    if m and name:
        kernels[name].append((int(m.group(1), 16), m.group(2), m.group(3)))


def slots(op):  # DESIGN.md section 4's dispatch-slot model: 64-bit-operand FP64 ops take 2 issue slots, IMAD.WIDE 2.5
    return 2.0 if op.split(".")[0] in ("DFMA", "DADD", "DMUL") else 2.5 if op.startswith("IMAD.WIDE") else 1.0


def show(label, ins):
    h = collections.Counter(op if full else op.split(".")[0] for _, op, _ in ins)
    print("  %-12s total %5d  slots %7.1f   %s" % (label, len(ins), sum(slots(op) for _, op, _ in ins),
                                                 ", ".join(f"{k} {v}" for k, v in h.most_common())))


for n, ins in kernels.items():
    if pat not in n:
        continue
    print(n, "total", len(ins))
    if not bodies:
        show("", ins)
        continue
    loops = []  # (start, end) address ranges of backward branches
    for addr, op, rest in ins:
        if op.startswith("BRA"):
            t = re.search(r"0x([0-9a-f]+)", rest)
            if t and int(t.group(1), 16) < addr:  # (the BRA-to-itself after EXIT is no loop)
                loops.append((int(t.group(1), 16), addr))
    inner = [l for l in loops if not any(o != l and l[0] <= o[0] and o[1] <= l[1] for o in loops)]
    groups = [[a for a in ins if lo <= a[0] <= hi] for lo, hi in inner]
    order = sorted(range(len(groups)), key=lambda i: -len(groups[i]))
    names = {}
    if len(order) >= 2:
        wide = lambda g: sum(1 for _, op, _ in g if op.startswith("IMAD.WIDE"))
        a, b = order[0], order[1]
        fr = a if wide(groups[a]) >= wide(groups[b]) else b
        names[fr] = "full_round"
        names[b if fr == a else a] = "partial_pair"
    inside = set()
    for i in order:
        show(names.get(i, "loop@%04x" % inner[i][0]), groups[i])
        inside.update(a for a, _, _ in groups[i])
    show("glue", [x for x in ins if x[0] not in inside])
