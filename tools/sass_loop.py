#!/usr/bin/env python
"""SASS instruction counts of a kernel's main loop, no GPU needed:

    python tools/sass_loop.py parallel-geometric-multigrid-for-poisson-problem_b200/csrc/kernels_fused.o 'k_crossILi4ELi2ELi2E'

For every function whose mangled name matches the regular expression: the whole kernel's size and opcode mix, then the body of
the LARGEST backward branch (the row loop of the streaming passes) -- its size, its full opcode mix, how many of its branches
leave it and how many other backward branches it contains.  Used for profiles/r3_* and r4_sass_k_cross_diet.txt.
"""
import collections
import os
import re
import subprocess
import sys

CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def opcode(ins):
    return re.sub(r"^@!?U?P\w+\s+", "", ins).split()[0]


def main():
    obj, pat = sys.argv[1], sys.argv[2]
    sass = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    for func in re.split(r"\n\s+Function : ", sass)[1:]:
        name = func.split("\n", 1)[0].strip()
        if not re.search(pat, name):
            continue
        ins = [(int(m.group(1), 16), m.group(2).strip()) for m in re.finditer(r"/\*([0-9a-f]{4,})\*/\s+([^;]*);", func)]
        target = {}
        for a, t in ins:
            m = re.search(r"0x([0-9a-f]+)", t) if opcode(t).startswith("BRA") else None
            if m:
                target[a] = int(m.group(1), 16)
        back = sorted(((a - b, b, a) for a, b in target.items() if b < a), reverse=True)
        print(name)
        print("  whole kernel: %d instructions" % len(ins), dict(collections.Counter(opcode(t) for _, t in ins).most_common()))
        if not back:
            continue
        _, lo, hi = back[0]
        body = [(a, t) for a, t in ins if lo <= a <= hi]
        leave = sum(1 for a, _ in body if a in target and not lo <= target[a] <= hi)
        inner = sum(1 for _, b, a in back[1:] if lo <= b and a <= hi)
        print("  loop 0x%x..0x%x: %d instructions, %d branches leave it, %d other backward branches inside" %
              (lo, hi, len(body), leave, inner))
        print("   ", dict(collections.Counter(opcode(t) for _, t in body).most_common()))


if __name__ == "__main__":
    main()
