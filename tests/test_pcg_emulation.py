"""The fused direction-operator pass of pmg_pcg on row slabs (csrc/kernel_pcg.cuh) executed WITHOUT a GPU under
tests/cpp/emu/host_emulation.h: whole levels n = 5 .. 1025 and the row-slab windows of 2, 4 and 8 ranks, with every z and p
row more than 1 row beyond the slab NaN and their Dirichlet ring NaN, for the first step (p = z) and a later one
(p = z + beta p).  p and A p are bit-identical to the oracle's direction update and apply_laplacian, every other element of
the output arrays (ring, padding, other rows) stays all-zero bits, the inputs keep their bits and the per-warp partial sums
add up to p . A p within 1e-14 relative (tests/cpp/test_pcg_emu.cpp)."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "parallel-geometric-multigrid-for-poisson-problem_b200")


def test_pcg_direction_apply_under_host_emulation(tmp_path):
    src = os.path.join(ROOT, "tests", "cpp", "test_pcg_emu.cpp")
    exe = str(tmp_path / "test_pcg_emu")
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-pthread", "-DPMG_HOST_EMULATION",
                    "-I" + os.path.join(ROOT, "tests", "cpp", "emu"), "-I" + os.path.join(PKG, "csrc"),
                    "-I" + os.path.join(ROOT, "include"), src, "-o", exe], check=True)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-2000:]
    assert "all bit-identical (36 runs)" in p.stdout and "MISMATCH" not in p.stdout
    assert p.stdout.count(": ok") == 36
