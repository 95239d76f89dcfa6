#!/usr/bin/env python
"""Writes the SASS of the tet walk's step loop (first crossing of tet_walk_fp64) with an instruction
census, from the built library (or another object given as the second argument) — no GPU needed:

    python scripts/sass_step_loop.py [kernel [library]] > profiles/r09_sass_step_loop.txt

The loop is found structurally: the first backward branch whose body holds exactly three global
loads, two or three of them LDG.E.ENL2.256 (the tet's Conn and Fields, the one new vertex; up to
r06 the two halves of the 64-byte cell and the vertex), and one MUFU.RCP64H (the divide of the exit
depth).
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    kernel = sys.argv[1] if len(sys.argv) > 1 else "tet_walk_fp64"
    so = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "course5_b200", "libc5gpu.so")
    names = subprocess.run(["cuobjdump", "-res-usage", so], capture_output=True, text=True).stdout
    res = {}
    fn = None
    for line in names.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            fn = m.group(1)
        elif fn and "REG:" in line:
            res[fn] = line.strip()
    full = next(n for n in res if kernel in n and "WalkParams" in n)
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", full, so], capture_output=True, text=True).stdout
    ins = []
    for line in sass.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2).strip()))
    addr_index = {a: i for i, (a, _) in enumerate(ins)}
    best = None
    for i, (a, text) in enumerate(ins):
        m = re.search(r"BRA\s+(?:P\d,\s*)?0x([0-9a-f]+)", text)
        if not m:
            continue
        target = int(m.group(1), 16)
        if target >= a or target not in addr_index:
            continue
        body = ins[addr_index[target]: i + 1]
        n256 = sum("LDG.E.ENL2.256" in t for _, t in body)
        nldg = sum(re.search(r"\bLDG\.", t) is not None for _, t in body)
        nrcp = sum("MUFU.RCP64H" in t for _, t in body)
        if nldg == 3 and n256 >= 2 and nrcp == 1:
            best = body
            break
    if best is None:
        raise SystemExit("step loop not found")
    print(f"# {kernel}: step loop of the first crossing (course5_b200/csrc/c5_walk.cu crossing_walk), "
          f"{len(best)} instructions, 0x{best[0][0]:x} .. 0x{best[-1][0]:x}")
    print(f"# {res[full]}")
    census = collections.Counter()
    for _, t in best:
        op = t.split()[1] if t.startswith("@") else t.split()[0]
        census[op.split(".")[0] + ("." + ".".join(op.split(".")[1:3]) if op.startswith(("LDG", "MUFU", "STG", "LDL", "STL")) else "")] += 1
    print("# census: " + ", ".join(f"{k} {v}" for k, v in census.most_common()))
    loads = [t for _, t in best if t.lstrip("@!P0123456789 ").startswith(("LDG", "LDL", "STL", "LDS"))]
    print(f"# memory instructions in the loop: {len(loads)}")
    for a, t in best:
        print(f"/*{a:04x}*/  {t} ;")


if __name__ == "__main__":
    main()
