"""The fused residual-restriction of the FMG set-up (csrc/kernel_residual_restrict.cuh) executed WITHOUT a GPU under
tests/cpp/emu/host_emulation.h: whole levels n = 5 .. 1025 and the row-slab windows of 2, 4 and 8 ranks, with every x row
more than 2 rows and every f row more than 1 row beyond the slab NaN, and an f with -0.0 and +-1e100 entries.  The coarse
right-hand side is bit-identical to the CPU oracle's residual followed by its restriction, every other element of the
coarse array (ring, other ranks' rows, padding) stays all-zero bits and the inputs keep their bits
(tests/cpp/test_residual_restrict_emu.cpp)."""
import os
import subprocess

import cpu_checkers as cc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200")


def test_residual_restrict_under_host_emulation(tmp_path):
    cc.load("orc")  # builds oracle/liboracle.so if needed
    src = os.path.join(ROOT, "tests", "cpp", "test_residual_restrict_emu.cpp")
    exe = str(tmp_path / "test_residual_restrict_emu")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-pthread", "-DPMG_HOST_EMULATION",
                    "-I" + os.path.join(ROOT, "tests", "cpp", "emu"), "-I" + os.path.join(PKG, "csrc"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", exe, "-L" + cc.ORACLE_DIR, "-loracle",
                    "-Wl,-rpath," + cc.ORACLE_DIR], check=True)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert "all bit-identical (18 runs)" in p.stdout and "MISMATCH" not in p.stdout
    assert p.stdout.count(": ok") == 18
