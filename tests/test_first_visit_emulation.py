"""The first visit of a coarse level (x == 0 on entry) on the fused engine, executed WITHOUT a GPU under
tests/cpp/emu/host_emulation.h: Pass A with its pointwise first sweep (an all-NaN iterate array, not read), with and without
the xb store, and Pass B reading xb or rebuilding it from f (an all-NaN xb array); n = 5 .. 1025, nu1, nu2 = 1 .. 3 and
(4, 4), omega = 1, 2/3, 0.8, 1.2, both prolongations, f with -0.0 and +-1e100 entries.  Every output bit-identical to the
CPU oracle, the padding of every output array all-zero bits, the skipped xb array untouched
(tests/cpp/test_first_visit_emu.cpp).  Dropping the pointwise sweep's +0 normalisation makes it fail (omega = 1, 1.2)."""
import os
import subprocess

import cpu_checkers as cc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200")


def test_first_visit_passes_under_host_emulation(tmp_path):
    cc.load("orc")  # builds oracle/liboracle.so if needed
    src = os.path.join(ROOT, "tests", "cpp", "test_first_visit_emu.cpp")
    exe = str(tmp_path / "test_first_visit_emu")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-pthread", "-DPMG_HOST_EMULATION",
                    "-I" + os.path.join(ROOT, "tests", "cpp", "emu"), "-I" + os.path.join(PKG, "csrc"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", exe, "-L" + cc.ORACLE_DIR, "-loracle",
                    "-Wl,-rpath," + cc.ORACLE_DIR], check=True)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert "all bit-identical (128 runs)" in p.stdout and "MISMATCH" not in p.stdout
    assert p.stdout.count(": ok") == 128
