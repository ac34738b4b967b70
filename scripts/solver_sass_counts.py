#!/usr/bin/env python
"""Instruction counts of the rank-64 one-warp solver (als_ws64_kernel's solver_role), read from the SASS of a built
library.  Runs on the CPU (cuobjdump, nm).

  python scripts/solver_sass_counts.py [path/to/libhals_b200.so]

The eight elimination loops (elim_block<JR>, JR = 0..7) are the loops of the kernel whose body holds both packed FMAs
(FFMA2) and a reciprocal (MUFU.RCP): one reciprocal per pivot step, so a body that runs two steps per iteration holds
two.  For each loop: instructions per pivot step, split into FFMA2, shared loads (LDS*), shared stores (STS*) and
everything else; then the dynamic elimination instructions per system (each body times its trip count, plus the
straight code between the loops: the column publish that opens blocks 1..7).  The two regions around the loops are
counted statically, both sides of every branch included: the stretch from the long-row slice copy loop to the first
elimination loop (the slice path's tail, the tile load from the hand-over slot, the implicit-mode Gram add and the
opening publish of block 0) and the one from the last elimination loop to the solver's row-loop branch (back
substitution and the row store)."""
import os
import re
import subprocess
import sys
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_LIB = os.path.join(ROOT, "hybrid-als-twotower-recommender_b200", "libhals_b200.so")
LINE = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")


def kernel_sass(lib):
    names = subprocess.run(["nm", "--defined-only", lib], capture_output=True, text=True, check=True).stdout.split()
    name = next(n for n in names if n.startswith("_ZN4hals4ws6415als_ws64_kernel"))
    out = subprocess.run(["cuobjdump", "-sass", "-fun", name, lib], capture_output=True, text=True, check=True).stdout
    ins = []
    for line in out.splitlines():
        m = LINE.match(line)
        if m:
            text = m.group(2)
            op = text.split()[1] if text.startswith("@") else text.split()[0]
            ins.append((int(m.group(1), 16), op, text))
    if not ins:
        sys.exit(f"no SASS for {name} in {lib}")
    return ins


def branch_target(op, text):
    if op.startswith("BRA") and not op.startswith("BRA.DIV"):
        m = re.search(r"0x([0-9a-f]+)\s*$", text)
        if m:
            return int(m.group(1), 16)
    return None


def klass(op):
    if op == "FFMA2":
        return "FFMA2"
    if op.startswith("LDS"):
        return "LDS"
    if op.startswith("STS"):
        return "STS"
    return "other"


def main():
    lib = sys.argv[1] if len(sys.argv) > 1 else DEFAULT_LIB
    ins = kernel_sass(lib)
    idx = {a: i for i, (a, _, _) in enumerate(ins)}
    loops = []                                   # (first index, last index) of each backward-branch loop
    for i, (a, op, text) in enumerate(ins):
        t = branch_target(op, text)
        if t is not None and t <= a and t in idx:
            loops.append((idx[t], i))
    inner = [(s, e) for s, e in loops if not any(s <= s2 and e2 < e for s2, e2 in loops)]   # no loop inside
    elim = [(s, e) for s, e in inner
            if any(ins[k][1] == "FFMA2" for k in range(s, e + 1)) and any(ins[k][1].startswith("MUFU.RCP") for k in range(s, e + 1))]
    elim.sort()
    if len(elim) != 8:
        sys.exit(f"expected 8 elimination loops, found {len(elim)}")

    print(f"# {os.path.relpath(lib, ROOT) if lib.startswith(ROOT) else lib}: als_ws64_kernel, solver elimination loops")
    print("| JR | instrs / pivot | FFMA2 | LDS | STS | everything else | steps / iteration | body |")
    print("|---|---|---|---|---|---|---|---|")
    dyn = Counter()
    tot_other = 0.0
    for jr, (s, e) in enumerate(elim):
        c = Counter(klass(ins[k][1]) for k in range(s, e + 1))
        steps = sum(ins[k][1].startswith("MUFU.RCP") for k in range(s, e + 1))
        n = e - s + 1
        per = {k: c[k] / steps for k in ("FFMA2", "LDS", "STS", "other")}
        tot_other += per["other"]
        fmt = lambda v: f"{v:.0f}" if v == int(v) else f"{v:.1f}"
        print(f"| {jr} | {fmt(n / steps)} | {fmt(per['FFMA2'])} | {fmt(per['LDS'])} | {fmt(per['STS'])} | "
              f"{fmt(per['other'])} | {steps} | {n} |")
        for k, v in c.items():
            dyn[k] += v * (8 // steps)
    gaps = Counter()
    for (s0, e0), (s1, _) in zip(elim, elim[1:]):
        for k in range(e0 + 1, s1):
            gaps[klass(ins[k][1])] += 1
    dyn_all = dyn + gaps
    static = sum(e - s + 1 for s, e in elim) + sum(gaps.values())
    print()
    print(f"'everything else' per pivot, mean over the 8 blocks: {tot_other / 8:.1f}")
    print(f"elimination per system (dynamic): {sum(dyn_all.values())} instructions = "
          + ", ".join(f"{dyn_all[k]} {k}" for k in ("FFMA2", "LDS", "STS", "other"))
          + f"  (loop bodies {sum(dyn.values())}, block openings 1..7 {sum(gaps.values())})")
    print(f"elimination code (static): {static} instructions")

    # tile load: from the end of the loop before loop 0 (the long-row slice copy) to loop 0
    s0 = elim[0][0]
    b = max(e for s, e in inner if e < s0)
    pre = Counter(ins[k][1] for k in range(b + 1, s0))
    # back substitution + store: from the end of loop 7 to the solver's row-loop branch (next backward branch)
    e7 = elim[-1][1]
    end = next((i for s, i in sorted(loops, key=lambda x: x[1]) if i > e7 and s < elim[0][0]), None)
    end = end if end is not None else next(i for i in range(e7 + 1, len(ins)) if ins[i][1].startswith("RET"))
    # out-of-line divergence paths (BRA.DIV targets) sit past the function's last instruction: not counted
    post = Counter(ins[k][1] for k in range(e7 + 1, end + 1))
    for label, c in (("slice-path tail + tile load + implicit Gram add + block-0 opening (static)", pre), ("back substitution + row store (static)", post)):
        top = ", ".join(f"{v} {k}" for k, v in c.most_common(8))
        print(f"{label}: {sum(c.values())} instructions; {top}")


if __name__ == "__main__":
    main()
