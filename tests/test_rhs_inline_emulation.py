"""The cross-cycle pass with its right-hand side generated in the row feed (csrc/kernels_fused.cu, SmemFeed with GEN_F)
executed WITHOUT a GPU under tests/cpp/emu/host_emulation.h: xb', the coarse right-hand side and the norm partials are
bit-identical to the same pass reading the stored f and to the CPU oracle, and the tables reproduce the stored array at
every position the pass reads, padding and sign of zero included (tests/cpp/test_rhs_inline_emu.cpp)."""
import os
import subprocess

import cpu_checkers as cc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200")


def test_generated_rhs_cross_pass_matches_stored_rhs_under_host_emulation(tmp_path):
    cc.load("orc")  # builds oracle/liboracle.so if needed
    src = os.path.join(ROOT, "tests", "cpp", "test_rhs_inline_emu.cpp")
    exe = str(tmp_path / "test_rhs_inline_emu")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-pthread", "-DPMG_HOST_EMULATION",
                    "-I" + os.path.join(ROOT, "tests", "cpp", "emu"), "-I" + os.path.join(PKG, "csrc"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", exe, "-L" + cc.ORACLE_DIR, "-loracle",
                    "-Wl,-rpath," + cc.ORACLE_DIR], check=True)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert "all bit-identical" in p.stdout and "MISMATCH" not in p.stdout
    assert p.stdout.count(": ok") == 7
