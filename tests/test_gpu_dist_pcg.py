"""pmg_pcg on row slabs on real hardware: launches tests/dist_check_pcg.py under torchrun on 2 GPUs, with the NVLink
peer-to-peer exchanges and with NCCL only (PMG_P2P=0), and on 3 GPUs where they are visible (slabs of unequal size, the
agglomerated level gathered to rank 0): the same step count as one GPU, history within 1e-10 relative, iterate within 1e-9
of its largest entry, a V-cycle afterwards bit-identical to one GPU -- and the two 2-GPU runs give bit-identical iterates.
Skipped on a single-GPU box -- the schedule itself is proven on CPU over gloo (test_dist_gloo_pcg.py) and the slab kernel
on one GPU (test_gpu_pcg_slabs.py)."""
import os
import re
import subprocess
import sys

import pytest

import pmg_b200 as pmg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
CASES = 8  # 2 sizes x 2 right-hand sides x precond 0 / 1


def _torchrun(ranks, port, **env):
    e = dict(os.environ, **env)
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks),
                           "--master-addr", "127.0.0.1", "--master-port", str(port),
                           os.path.join(ROOT, "tests", "dist_check_pcg.py"), "1025", "4097"],
                          capture_output=True, text=True, timeout=1200, env=e)


def test_pcg_two_gpus_match_one_gpu_with_and_without_p2p():
    if pmg.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    digests = []
    for p2p, port in (("1", 29561), ("0", 29562)):
        p = _torchrun(2, port, PMG_P2P=p2p)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        assert "FAIL" not in p.stdout and p.stdout.count(" OK") == CASES
        digests.append(re.findall(r"digest=(\w+)", p.stdout))
    assert len(digests[0]) == CASES and digests[0] == digests[1], digests


def test_pcg_three_gpus_match_one_gpu():
    if pmg.device_count() < 3:
        pytest.skip("needs 3 GPUs")
    p = _torchrun(3, 29563)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "FAIL" not in p.stdout and p.stdout.count(" OK") == CASES
