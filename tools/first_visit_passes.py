#!/usr/bin/env python
"""Times the two passes of a first visit (x == 0 on entry) of one level alone, with CUDA events over many launches
(pmg_bench_pass): Pass A with x == 0 (which = 3) and Pass B without the norm (which = 2), on levels n = 8193, 4097 and
2049 (level 0 of a solver of that size, V(2,2), omega = 2/3, sine right-hand side).  PMG_LIB=<path> times another build
of libpmg.so, so that two builds can be compared on one box.  One JSON line per level: the best of 3 averages of `reps`
launches each.

    python tools/first_visit_passes.py [reps]
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pmg_b200 as pmg  # noqa: E402

if os.environ.get("PMG_LIB"):
    sys.modules["_pmg_b200_pkg"].LIB_PATH = os.path.abspath(os.environ["PMG_LIB"])


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    for n in (8193, 4097, 2049):
        s = pmg.Solver(n, omega=2.0 / 3.0)
        s.set_rhs_sine()
        row = {"n": n, "reps": reps}
        for name, which in (("pass_a_x0", 3), ("pass_b", 2)):
            s.bench_pass(which, 0, 20)  # warm-up
            row[name + "_us"] = round(1e3 * min(s.bench_pass(which, 0, reps) for _ in range(3)), 2)
        print(json.dumps(row), flush=True)
        s.close()


if __name__ == "__main__":
    main()
