"""Pass B with the coarse up-exchange prologue of the deep-sweep slab schedule (k_up with UPX, csrc/kernels_fused.cu)
executed WITHOUT a GPU under tests/cpp/emu/host_emulation.h, on 2-4 row slabs side by side: every (nu1, nu2) with a 3 or
4, the finest level and a coarser one, both prolongations, omega 2/3 and 1, chunks of 4 rows (148 SMs) and tall chunks.
The coarse rows the prologue must copy are NaN until it copies them, and the emulator runs the warps one after another in
index order, so a warp that reads a copied row without waiting for and copying it reads NaN.  x is bit-identical to the
oracle, nothing outside the pass's rows changes -- padding bits included -- and every epoch is published
(tests/cpp/test_up_exchange_emu.cpp)."""
import os
import subprocess

import cpu_checkers as cc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200")


def test_up_exchange_prologue_under_host_emulation(tmp_path):
    cc.load("orc")  # builds oracle/liboracle.so if needed
    src = os.path.join(ROOT, "tests", "cpp", "test_up_exchange_emu.cpp")
    exe = str(tmp_path / "test_up_exchange_emu")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-pthread", "-DPMG_HOST_EMULATION",
                    "-I" + os.path.join(ROOT, "tests", "cpp", "emu"), "-I" + os.path.join(PKG, "csrc"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", exe, "-L" + cc.ORACLE_DIR, "-loracle",
                    "-Wl,-rpath," + cc.ORACLE_DIR], check=True)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert "all bit-identical (48 runs)" in p.stdout and "MISMATCH" not in p.stdout
    assert p.stdout.count(": ok") == 48
