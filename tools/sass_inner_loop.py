#!/usr/bin/env python3
"""Dumps the LF-step loop of search_kernel from the built object (cuobjdump -sass, no GPU needed) with per-class
instruction counts, into a markdown file under profiles/ (VERDICT r1 item 7 / next-round item 5).

The loop is found structurally: it is the code between the `VOTE.ANY` that opens the step (no lane has a read ->
leave) and the backward branch that closes it; the rare warp-cooperative paths (cluster children, terminator window)
sit behind a forward branch inside it and are reported separately.

  python tools/sass_inner_loop.py [--md profiles/r2_search_kernel_sass.md]
"""
import argparse
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "rowbowt_b200", "csrc", "build", "kernels.o")
CLASSES = [
    ("decode: IDP.2A (two-way dot products)", r"^IDP"),
    ("decode: VIMNMX.U16x2 (packed mins)", r"^VIMNMX"),
    ("logic: LOP3 / SHF / PRMT / SEL / POPC", r"^(LOP3|SHF|PRMT|SEL|POPC|FLO|BREV)"),
    ("integer: IMAD / IADD3 / LEA / VIADD / MOV", r"^(IMAD|IADD3|LEA|VIADD|MOV|CS2R|IABS)"),
    ("global loads LDG", r"^LDG"),
    ("shared / constant loads LDS, LDC, LDCU", r"^(LDS|LDC|LDCU|ULDC)"),
    ("stores / atomics", r"^(STG|STS|ATOM|RED|STL|LDL)"),
    ("predicates ISETP / PLOP3", r"^(ISETP|PLOP3|P2R|R2P)"),
    ("warp ops VOTE / SHFL / REDUX / MATCH", r"^(VOTE|SHFL|REDUX|MATCH|WARPSYNC)"),
    ("control BRA / BSSY / BSYNC / EXIT", r"^(BRA|BSSY|BSYNC|EXIT|CALL|RET|NOP|BAR)"),
    ("uniform datapath U*", r"^(U[A-Z0-9]+|S2UR|R2UR)"),
]


def sass_of(variant):
    names = subprocess.run(["cuobjdump", "-sass", OBJ], capture_output=True, text=True).stdout
    m = re.search(r"Function : (\S*search_kernel%s\S*)" % variant, names)
    if not m:
        raise SystemExit("kernel variant %s not found" % variant)
    txt = subprocess.run(["cuobjdump", "-sass", "-fun", m.group(1), OBJ], capture_output=True, text=True).stdout
    ins = []
    for ln in txt.split("\n"):
        mm = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);", ln)
        if mm:
            body = re.sub(r"^@!?U?P\w+\s+", "", mm.group(2).strip())
            ins.append((int(mm.group(1), 16), mm.group(2).strip(), body.split()[0].split(".")[0], body))
    return ins


def classify(ins):
    c = collections.Counter()
    for _, _, op, body in ins:
        for name, rx in CLASSES:
            if re.match(rx, body):
                c[name] += 1
                break
        else:
            c["other: " + op] += 1
    return c


def branch_target(full):
    mm = re.search(r"BRA\S*\s+(?:\w+,\s*)?0x([0-9a-f]+)", full)
    return int(mm.group(1), 16) if mm else None


def loop_parts(ins, anchor="IDP", lead=0x200):
    """Splits the outer loop of search_kernel into (refill, common step path, rare path) by structure:
    the loop = the longest backward branch; the step starts at the last branch-join at least `lead` bytes before the first
    `anchor` instruction of the ranks (IDP.2A on the run-length lines, POPC on the plain lines; the read refill sits in
    front of it); the rare block is what the first forward branch after the decode's VOTE skips."""
    best = None
    first_exit = min([x[0] for x in ins if x[2] == "EXIT"] + [1 << 30])      # the loop ends before the kernel's epilogue
    for addr, full, op, body in ins:
        if addr > first_exit:
            break
        tgt = branch_target(full)
        if op == "BRA" and "BRA.DIV" not in full and tgt is not None and tgt < addr - 0x100 and (best is None or addr - tgt > best[1] - best[0]):
            best = (tgt, addr)
    start, end = best
    loop = [x for x in ins if start <= x[0] <= end]
    first_line = next(x[0] for x in loop if x[2] == "LDG" and ".256" in x[1])     # the step's first directory line load
    idp = [x[0] for x in loop if x[2] == anchor and x[0] > first_line]
    first_idp = idp[0]
    last_core_idp = first_idp
    for a in idp:                                              # the first dense run of IDPs = the two ranks of the common path
        if a - last_core_idp <= 0x280:
            last_core_idp = a
    joins = sorted({branch_target(x[1]) for x in loop if x[2] == "BRA" and branch_target(x[1]) is not None and branch_target(x[1]) > x[0]})
    step_start = max([j for j in joins if j <= first_idp - lead] + [start])
    vote = next(x[0] for x in loop if x[0] > last_core_idp and x[2] == "VOTE")
    rb = next(x for x in loop if x[0] > vote and x[2] == "BRA" and branch_target(x[1]) and branch_target(x[1]) > x[0])
    rare = (rb[0], branch_target(rb[1]))
    refill = [x for x in loop if x[0] < step_start]
    rare_ins = [x for x in loop if rare[0] < x[0] < rare[1]]
    common = [x for x in loop if x[0] >= step_start and not (rare[0] < x[0] < rare[1])]
    return (start, end, step_start, rare), refill, common, rare_ins


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--md", default=os.path.join(ROOT, "profiles", "r2_search_kernel_sass.md"))
    a = ap.parse_args()
    out = ["# search_kernel: SASS of the LF-step loop (sm_100a, `cuobjdump -sass rowbowt_b200/csrc/build/kernels.o`)", "",
           "Per-class instruction counts of ONE pass through the step loop (one LF step for all 32 lanes of a warp).  For the toehold",
           "variants the `common path` column also holds the block of the third rank, which runs in about one warp step in six.",
           "`common path` = what every warp step executes; `rare path` = the forward-branched block that runs only when some lane's",
           "rank position lies inside a collapsed variant cluster / the terminator window (warp-cooperative child-line walk).", ""]
    for variant, label, anchor, lead in (("ILb0ELi7ELb0EE", "count, layout 7", "POPC", 0x100),
                                         ("ILb1ELi7ELb0EE", "toehold (-s), layout 7", "POPC", 0x100),
                                         ("ILb0ELi5ELb0EE", "count, layout 5", "IDP", 0x200),
                                         ("ILb1ELi5ELb0EE", "toehold (-s), layout 5", "IDP", 0x200),
                                         ("ILb0ELi4ELb0EE", "count, layout 4", "IDP", 0x200)):
        ins = sass_of(variant)
        (start, end, step_start, rare), refill, common, rare_ins = loop_parts(ins, anchor, lead)
        out += ["## %s — `search_kernel<%s>`" % (label, variant), "",
                "loop 0x%04x..0x%04x; LF step from 0x%04x: **%d instructions on the common path** of a step, %d in the rare block "
                "(0x%04x..0x%04x), %d in the read refill in front of the step (runs when a quarter of the warp is idle)" % (
                    start, end, step_start, len(common), len(rare_ins), rare[0], rare[1], len(refill)), "",
                "| class | common path | rare block | refill |", "|---|---:|---:|---:|"]
        cc, rc, fc = classify(common), classify(rare_ins), classify(refill)
        for name in sorted(set(cc) | set(rc) | set(fc), key=lambda k: -cc.get(k, 0)):
            out.append("| %s | %d | %d | %d |" % (name, cc.get(name, 0), rc.get(name, 0), fc.get(name, 0)))
        out.append("")
        if variant in ("ILb0ELi7ELb0EE", "ILb0ELi5ELb0EE"):
            out += ["<details><summary>common path, full listing</summary>", "", "```"]
            out += ["/*%04x*/ %s ;" % (x[0], x[1]) for x in common]
            out += ["```", "", "</details>", ""]
    open(a.md, "w").write("\n".join(out) + "\n")
    print("\n".join(out[:60]))


if __name__ == "__main__":
    main()
