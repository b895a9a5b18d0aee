"""GPU tests of the sharded paths (SURVEY §8e, ADVICE r1): `register_pair_sharded` (cost rows to the owner through
the peer-mapped window and through dist.gather) and `register_all_pairs` (unequal specimen sizes, 3 registrations in
flight, shared work counter) reproduce the single-GPU pipeline.  tools/dist_check.py does the work: in this process on
one GPU, and under torchrun with NCCL on two when the box has them."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(cmd):
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "DIST_CHECK_OK" in p.stdout, p.stdout[-3000:] + "\n" + p.stderr[-3000:]
    return p.stdout


def test_sharded_paths_single_gpu():
    print(_run([sys.executable, "tools/dist_check.py"]))


def test_sharded_paths_two_gpus_nccl():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (on one GPU, test_sharded_paths_single_gpu covers world = 1)")
    print(_run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                "--master-addr", "127.0.0.1", "--master-port", "29533", "tools/dist_check.py"]))
