"""The cross-cycle pass (csrc/kernels_fused.cu, k_cross) at the edges of the level, executed WITHOUT a GPU under
tests/cpp/emu/host_emulation.h: a non-zero Dirichlet ring with -0.0 and values of magnitude 1e100, both prolongations, wide
and narrow shapes, stored and generated f, row slabs on 2-4 ranks; every output bit-identical to the CPU oracle and the
padding of every output array still all-zero bits (tests/cpp/test_cross_edges_emu.cpp)."""
import os
import subprocess

import cpu_checkers as cc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200")


def test_cross_pass_edges_and_padding_under_host_emulation(tmp_path):
    cc.load("orc")  # builds oracle/liboracle.so if needed
    src = os.path.join(ROOT, "tests", "cpp", "test_cross_edges_emu.cpp")
    exe = str(tmp_path / "test_cross_edges_emu")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-pthread", "-DPMG_HOST_EMULATION",
                    "-I" + os.path.join(ROOT, "tests", "cpp", "emu"), "-I" + os.path.join(PKG, "csrc"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", exe, "-L" + cc.ORACLE_DIR, "-loracle",
                    "-Wl,-rpath," + cc.ORACLE_DIR], check=True)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert "all bit-identical" in p.stdout and "MISMATCH" not in p.stdout
    assert p.stdout.count(": ok") == 15
    assert p.stdout.count("slabs") == 4
