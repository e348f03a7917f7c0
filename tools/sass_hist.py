#!/usr/bin/env python
"""Opcode histogram of the hot loops of one kernel (cuobjdump -sass of an object file): the loops are the largest
backward branches; counts are per loop body and per row (body / rows_per_body).  ALU-pipe opcodes are summed, since that
pipe bounds the sweep kernels.   usage: sass_hist.py <object> <mangled-kernel-substring> [rows_per_body] [min_bytes]

Static counts include code a row rarely runs.  The "common path" line walks one pass of the loop instead: it falls
through conditional branches, but jumps over the blocks a row skips in the common case -- a spin wait (a block with
NANOSLEEP or an exit from the loop that loads no row data) and the in-row scan's long-chain stages (a branch right
after a VOTE) -- and it does not follow BRA.DIV (taken only when the warp has diverged)."""
import collections
import re
import subprocess
import sys

ALU = {"LOP3", "LEA", "SHF", "ISETP", "IADD3", "SEL", "VIADD", "PLOP3", "VIMNMX", "VIADDMNMX", "PRMT", "POPC", "FLO", "IABS", "BMSK", "SGXT", "LOP"}


def main(obj, sub, rows=3, min_bytes=0x2000):
    names = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    fn = None
    for m in re.finditer(r"Function : (\S+)", names):
        if sub in m.group(1):
            fn = m.group(1)
            break
    if not fn:
        sys.exit("kernel not found")
    txt = subprocess.run(["cuobjdump", "-sass", "-fun", fn, obj], capture_output=True, text=True).stdout
    ins = []
    for l in txt.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
        if m:
            ins.append((int(m.group(1), 16), re.sub(r"^@!?U?P\d+\s+", "", m.group(2).strip()), m.group(2).strip().startswith("@")))
    print(fn, len(ins), "instructions")
    loops = []
    for a, t, pred in ins:
        m = re.search(r"BRA\S*\s+(?:!?U?P\d+,\s*|UR\d+,\s*)?0x([0-9a-f]+)", t)
        if m and pred and int(m.group(1), 16) < a and min_bytes <= a - int(m.group(1), 16) < 0x8000:
            loops.append((int(m.group(1), 16), a))
    for lo, hi in loops:
        c = collections.Counter(t.split()[0].split(".")[0] for a, t, _ in ins if lo <= a <= hi)
        tot = sum(c.values())
        alu = sum(v for k, v in c.items() if k in ALU)
        print(f"loop {lo:#x}..{hi:#x}: {tot} instr = {tot / rows:.1f} per row, ALU pipe {alu} = {alu / rows:.1f} per row")
        print("   " + "  ".join(f"{k} {v / rows:.1f}" for k, v in c.most_common(14)))
        path = common_path(ins, lo, hi)
        c = collections.Counter(t.split()[0].split(".")[0] for t in path)
        tot, alu = sum(c.values()), sum(v for k, v in c.items() if k in ALU)
        special = {"BRA.DIV": sum(t.startswith("BRA.DIV") for t in path),
                   "UMOV 0xffffffff": sum(t.startswith("UMOV") and t.endswith("0xffffffff") for t in path),
                   "CS2R SRZ": sum(t.startswith("CS2R") and t.endswith("SRZ") for t in path)}
        print(f"   common path: {tot / rows:.1f} instr per row, ALU pipe {alu / rows:.1f} per row;  "
              + "  ".join(f"{k} {v / rows:.1f}" for k, v in special.items()))
        print("   " + "  ".join(f"{k} {v / rows:.1f}" for k, v in c.most_common(14)))


def common_path(ins, lo, hi):
    """instructions (predicates stripped) of one pass through the loop lo..hi in the common case"""
    at = {a: i for i, (a, _, _) in enumerate(ins)}
    i, path = at[lo], []
    while ins[i][0] <= hi and len(path) < 20000:
        a, t, pred = ins[i]
        path.append(t)
        m = re.match(r"BRA(\.\S+)?\s+(?:!?U?P\d+,\s*|UR\d+,\s*)?0x([0-9a-f]+)", t)
        if a == hi:
            break
        if not m:
            i += 1
            continue
        tgt = int(m.group(2), 16)
        if m.group(1) == ".DIV":
            i += 1
        elif not pred:
            i = at[tgt]
        elif tgt > a and any("VOTE" in ins[k][1] for k in range(max(0, i - 4), i)):
            i = at[tgt]
        elif tgt > a and tgt in at:
            block = [x[1] for x in ins[i + 1:at[tgt]]]
            exits = any((b := re.search(r"BRA\s+0x([0-9a-f]+)", x)) and int(b.group(1), 16) > hi for x in block)
            rows = any(re.match(r"LDG\S*\s+R\d+, desc\[\w+\]\[R\d+\.64\+0x", x) or x.startswith(("LDG.E.64", "LDG.E.128"))
                       for x in block)      # row data: vector loads or loads at an offset from a row pointer
            i = at[tgt] if not rows and (exits or any(x.startswith("NANOSLEEP") for x in block)) else i + 1
        else:
            i += 1
    return path


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2], *(int(x, 0) for x in sys.argv[3:]))
