"""Instruction mix of the DP step of every packed-half scan instantiation, read from a built object's SASS:
    python tools/sass_step_mix.py soundsym_b200/csrc/_obj/dtw_h2.o [> profiles/...]

Each function of the object whose name contains `k_dtw_scan_h2` is split into basic blocks (a block starts at a branch target
or after a branch), and every block that holds a VHMNMX is printed with its mix:
  band   VHMNMX (the three-input min) and HADD2 / HFMA2 (the add; the compiler alternates the two forms): 2 per half2 cell
  moves  register moves, MOV / IMAD.MOV (register copies and re-materialised constants alike)
  other  everything else (TMEM loads and waits, barriers, address arithmetic, the loop's compare and branch, capture picks)
`loop` marks a block that ends in a backward branch (to its own start or to the barrier wait in front of it): the steps
that run several times in a row, the capture-free ones and the capture steps at a tile's end. NG is the
band's 4-column groups, VHMNMX / (8 NB) for a two-row step; a block with half of that is the odd last row of a tile, one
with extra `other` the capture steps at a tile's end. The band alone needs 2 instructions per half2 cell."""
import collections
import re
import subprocess
import sys

INSN = re.compile(r"^\s+/\*([0-9a-f]{4,6})\*/\s+(@!?U?P[T0-9]+\s+)?([A-Z0-9_]+(?:\.[A-Z0-9_x]+)*)\s*([^;]*);")
BRANCH = ("BRA", "BRX", "JMP", "JMX", "EXIT", "RET", "CALL", "BREAK", "KILL")


def blocks(body):
    ins = []
    for l in body.split("\n"):
        m = INSN.match(l)
        if m:
            ins.append((int(m.group(1), 16), m.group(3), m.group(4), bool(m.group(2))))
    leaders = {ins[0][0]} if ins else set()
    for i, (addr, op, args, _) in enumerate(ins):
        if op.split(".")[0] in BRANCH:
            t = re.search(r"0x([0-9a-f]+)\s*$", args.strip())
            if t and op.split(".")[0] in ("BRA", "JMP"):
                leaders.add(int(t.group(1), 16))
            if i + 1 < len(ins):
                leaders.add(ins[i + 1][0])
    out, cur = [], []
    for insn in ins:
        if insn[0] in leaders and cur:
            out.append(cur)
            cur = []
        cur.append(insn)
    if cur:
        out.append(cur)
    return out


def mix(block):
    c = collections.Counter()
    for _, op, _, _ in block:
        base = op.split(".")[0]
        if base == "VHMNMX":
            c["vhmnmx"] += 1
        elif base in ("HADD2", "HFMA2"):
            c["add"] += 1
        elif base == "MOV" or op.startswith("IMAD.MOV"):
            c["moves"] += 1
        else:
            c["other"] += 1
    return c


def main(paths):
    for obj in paths:
        txt = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
        print("==== %s" % obj)
        for f in re.split(r"\n\s+Function : ", txt)[1:]:
            name = f.split("\n")[0].strip()
            if "k_dtw_scan_h2" not in name:
                continue
            demangled = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
            m = re.search(r"<(\d+), (\d+), (true|false)>", demangled)
            nb = int(m.group(2)) if m else 1
            print("%s" % demangled)
            print("   %-13s %5s %6s %6s %6s %6s %6s  %s" % ("block", "NG", "VHMNMX", "add", "moves", "other", "total", ""))
            for b in blocks(f):
                c = mix(b)
                if not c["vhmnmx"]:
                    continue
                last_op, last_args = b[-1][1], b[-1][2]
                t = re.search(r"0x([0-9a-f]+)\s*$", last_args.strip())
                loop = last_op.startswith("BRA") and t is not None and int(t.group(1), 16) <= b[0][0]
                ng = c["vhmnmx"] / (8.0 * nb)
                print("   %05x-%05x %5s %6d %6d %6d %6d %6d  %s" % (b[0][0], b[-1][0], ("%g" % ng), c["vhmnmx"], c["add"], c["moves"], c["other"],
                                                             sum(c.values()), "loop" if loop else ""))


if __name__ == "__main__":
    main(sys.argv[1:])
