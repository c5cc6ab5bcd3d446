"""PMG_CYCLE_FMG on row slabs on real hardware: launches tests/dist_check_fmg.py under torchrun on 2 GPUs, with the
NVLink peer-to-peer exchanges and with NCCL only (PMG_P2P=0): pass and FMG-then-V solve bit-identical to one GPU, norms and
histories to 1e-12.  Where the slabs of the first agglomerated level are unequal (PMG_COARSE_GATHER=1 on 2 GPUs; 3 ranks
where 3 GPUs are visible) every rank must get PMG_ERR_UNSUPPORTED and exit cleanly.  Skipped on a single-GPU box -- the
schedule itself is proven on CPU over gloo (test_dist_gloo_fmg.py) and the slab kernel on one GPU (test_gpu_fmg_slabs.py)."""
import os
import subprocess
import sys

import pytest

import pmg_b200 as pmg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _torchrun(ranks, port, args, **env):
    e = dict(os.environ, **env)
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks),
                           "--master-addr", "127.0.0.1", "--master-port", str(port),
                           os.path.join(ROOT, "tests", "dist_check_fmg.py")] + args,
                          capture_output=True, text=True, timeout=1200, env=e)


@pytest.mark.parametrize("p2p", ["1", "0"])
def test_fmg_two_gpus_match_one_gpu(p2p):
    if pmg.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    p = _torchrun(2, 29551 if p2p == "1" else 29552, ["1025", "4097"], PMG_P2P=p2p)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "FAIL" not in p.stdout and p.stdout.count(" OK") == 32


def test_fmg_unequal_slabs_refused_on_every_rank():
    if pmg.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    p = _torchrun(2, 29553, ["--expect-unsupported"], PMG_COARSE_GATHER="1")
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "refused at cycle on every rank: OK" in p.stdout


def test_fmg_three_ranks_refused_on_every_rank():
    if pmg.device_count() < 3:
        pytest.skip("needs 3 GPUs")
    p = _torchrun(3, 29554, ["--expect-unsupported"])
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "unsupported ranks=3" in p.stdout and "on every rank: OK" in p.stdout
