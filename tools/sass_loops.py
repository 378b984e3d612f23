#!/usr/bin/env python3
"""Static instruction counts of the loops of one kernel, from `cuobjdump -sass` output.

usage: cuobjdump -sass zipnn_b200/csrc/libzipnn_b200.so > lib.sass
       python tools/sass_loops.py lib.sass k_encode_write_warpILi2 [min_instructions]

A loop is the span from the target of a backward branch to that branch, both included.  For each loop of
at least `min_instructions` (default 60) it prints the number of instructions and how many of them are
branches (BRA), convergence markers (BSSY / BSYNC), shared-memory reductions (ATOMS), shared loads and
stores, shuffles and global/generic stores.  The innermost loop that holds the tile work of
k_encode_write_warp is the one DESIGN.md §3.3 quotes."""
import re
import sys


def main():
    path, kernel = sys.argv[1], sys.argv[2]
    min_len = int(sys.argv[3]) if len(sys.argv) > 3 else 60
    txt = open(path).read()
    for f in re.split(r"\n\s*Function : ", txt)[1:]:
        name = f.split("\n", 1)[0].strip()
        if kernel not in name:
            continue
        ins = [(int(m.group(1), 16), m.group(2)) for m in re.finditer(r"/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", f)]
        print(f"{name}: {len(ins)} instructions")
        for addr, op in ins:
            m = re.search(r"\bBRA(?:\.\w+)*\s+(?:\w+,\s*)?0x([0-9a-f]+)", op)
            if not m or int(m.group(1), 16) >= addr:
                continue
            tgt = int(m.group(1), 16)
            span = [o for a, o in ins if tgt <= a <= addr]
            if len(span) < min_len:
                continue

            def cnt(pat):
                return sum(1 for o in span if re.search(pat, o))
            print(f"  loop {tgt:#06x}..{addr:#06x}: {len(span)} instructions, {cnt(r'\bBRA\b')} BRA, "
                  f"{cnt(r'BSSY|BSYNC')} BSSY/BSYNC, {cnt(r'\bATOMS')} ATOMS, {cnt(r'\bLDS')} LDS, {cnt(r'\bSTS')} STS, "
                  f"{cnt(r'SHFL')} SHFL, {cnt(r'\bST\.|\bSTG')} ST/STG")


if __name__ == "__main__":
    main()
