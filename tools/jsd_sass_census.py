"""SASS census of jsd_tile_kernel<float>'s three chunk loops (V0, V1, V2), per dimension.

    python tools/jsd_sass_census.py [OBJ_OR_SO]      (default: phyloligo_b200/lib/obj/po_jsd.o)

Runs cuobjdump -sass (no GPU needed), finds the loop bodies (the code between a backward branch's
target and the branch), and for each prints the instruction count per opcode and the 32-bit register
source reads per lane: an F32x2 operand reads two registers, a .F32 broadcast operand one, any other
register source one (64-bit LDS/LDL address operands count one).  Sources marked .reuse are counted
apart: they are served by the operand reuse cache, not the register file.  The loops are unrolled
JSD_UNROLL (2) times; the counts are divided by the dimensions one pass covers.  A loop is V0 when it
has 40 FFMA2 per dimension, V1 at 56; V2 is the loop with the warp vote.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNEL = "_ZN2po15jsd_tile_kernelIfEEvNS_9JsdParamsE"
UNROLL = 2

LINE = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def kernel_sass(path):
    out = subprocess.run(["cuobjdump", "-sass", "-fun", KERNEL, path], capture_output=True, text=True, check=True).stdout
    ins = []
    for m in LINE.finditer(out):
        ins.append((int(m.group(1), 16), m.group(2)))
    return ins


def reads(text):
    """(register-file reads, reuse hits) of one instruction's sources."""
    body = re.sub(r"^@!?U?P\w+\s+", "", text)
    parts = body.split(None, 1)
    if len(parts) < 2:
        return 0, 0
    op, args = parts
    ops = [a.strip() for a in args.split(",")]
    srcs = ops[1:] if not op.startswith(("ST", "BRA", "BAR", "SYNCS", "RED", "ATOM")) else ops
    rf = hit = 0
    for a in srcs:
        for r in re.finditer(r"-?\|?(R\d+)((?:\.\w+)*)", a):
            mods = r.group(2)
            n = 2 if "F32x2" in mods else 1
            if ".64" in op and "[" in a:
                n = 1
            if ".reuse" in mods:
                hit += n
            else:
                rf += n
    return rf, hit


def census(ins):
    loops = []
    for addr, text in ins:
        m = re.search(r"BRA(?:\.U)?\s+(?:!?U?P\w+,\s*)?0x([0-9a-f]+)", text)
        if m and int(m.group(1), 16) < addr:
            lo = int(m.group(1), 16)
            body = [t for a, t in ins if lo <= a <= addr]
            # innermost loops only: the chunk loop around them waits on the stage's mbarrier
            if sum(t.startswith("FFMA2") for t in body) >= 40 and not any(t.startswith("SYNCS") for t in body):
                loops.append(body)
    res = []
    for body in loops:
        ops = collections.Counter()
        rf = hit = 0
        for t in body:
            op = re.sub(r"^@!?U?P\w+\s+", "", t).split()[0]
            ops[op] += 1
            a, b = reads(t)
            rf += a
            hit += b
        ffma2 = ops["FFMA2"] / UNROLL
        name = "V2" if any(k.startswith("VOTE") or k.startswith("REDUX") or k.startswith("CREDUX") for k in ops) else (
            "V0" if ffma2 <= 44 else "V1")
        res.append((name, ops, rf / UNROLL, hit / UNROLL))
    return res


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "phyloligo_b200", "lib", "obj", "po_jsd.o")
    for name, ops, rf, hit in sorted(census(kernel_sass(path)), key=lambda r: r[0]):
        per = {k: v / UNROLL for k, v in sorted(ops.items(), key=lambda kv: -kv[1])}
        print("%s  register-file reads/dim %.1f  reuse hits/dim %.1f" % (name, rf, hit))
        print("    " + "  ".join("%s %g" % kv for kv in per.items()))


if __name__ == "__main__":
    main()
