"""The deep-sweep slab schedule (3 or 4 pre/post-smoothing sweeps) on real hardware: launches
tests/dist_check_deep_sweeps.py under torchrun on 2 GPUs, with the NVLink peer-to-peer exchanges and with NCCL only
(PMG_P2P=0): V-, W- and F-cycles, a solve, FMG-then-V and PCG bit-identical to (PCG: within tolerance of) one GPU, the
refusal of nu = 0 / 5 on every rank -- and the two 2-GPU runs give bit-identical iterates.  On 3 GPUs, where they are
visible: the refusals on every rank (a row partition over 3 ranks does not nest across levels, which pmg_create rejects
at every N).  Skipped on a single-GPU box: the schedule itself is proven on CPU over gloo (test_dist_gloo_deep_sweeps.py)
and the slab kernels on one GPU (test_gpu_deep_sweep_slabs.py)."""
import os
import re
import subprocess
import sys

import pytest

import pmg_b200 as pmg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _torchrun(ranks, port, **env):
    e = dict(os.environ, **env)
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks),
                           "--master-addr", "127.0.0.1", "--master-port", str(port),
                           os.path.join(ROOT, "tests", "dist_check_deep_sweeps.py"), "1025", "4097"],
                          capture_output=True, text=True, timeout=1800, env=e)


def test_deep_sweeps_two_gpus_match_one_gpu_with_and_without_p2p():
    if pmg.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    digests = []
    for p2p, port in (("1", 29571), ("0", 29572)):
        p = _torchrun(2, port, PMG_P2P=p2p)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        assert "FAIL" not in p.stdout
        digests.append(re.findall(r"digest=(\w+)", p.stdout))
    assert digests[0] == digests[1], digests


def test_deep_sweeps_three_gpus_match_one_gpu():
    if pmg.device_count() < 3:
        pytest.skip("needs 3 GPUs")
    p = _torchrun(3, 29573)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "FAIL" not in p.stdout
