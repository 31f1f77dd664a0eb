"""Multi-GPU parity: one tree cut over 2 GPUs, gathered solution vs the oracle's direct solve of
the whole network (tests/dist_check.py under torchrun).  The 2-GPU cases are skipped on single-GPU boxes; the
one-GPU cases run the same partition and the split-phase kernels with both ranks on cuda:0 and gloo collectives."""

import pathlib
import subprocess
import sys

import pytest

from tests import helpers

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("args", [
    ("11", "1", "64", "tree", "peer"),       # in-kernel NVLink exchange (fused kernels)
    ("11", "1", "64", "tree", "nccl"),       # split phases around torch.distributed all-reduces
    ("9", "4", "32", "tree", "auto"),        # refined edges (4 cells per edge): fused kernels with array staging
    ("10", "1", "64", "arterial", "peer"),   # BASELINE configs[3]: radius-dependent R, f != 0
    ("8", "4", "32", "arterial", "peer"),
    ("8", "4", "32", "arterial", "nccl"),
])
def test_single_tree_partition_two_gpus(args):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(helpers.free_port()), str(ROOT / "tests" / "dist_check.py"), *args]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "-> OK" in out.stdout


@pytest.mark.parametrize("args,world", [
    (("11", "1", "64", "tree", "nccl"), 2),
    (("8", "4", "32", "arterial", "nccl"), 2),
    (("10", "1", "32", "arterial", "nccl"), 4),
])
def test_single_tree_partition_ranks_sharing_one_gpu(args, world):
    """Distributed parity that a single-GPU box can run: ``world`` ranks on cuda:0, host-driven exchange over
    gloo; the gathered solution against the oracle's direct solve of the whole network."""
    import os

    env = dict(os.environ, NXFX_DIST_ONE_GPU="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(helpers.free_port()), str(ROOT / "tests" / "dist_check.py"), *args]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "-> OK" in out.stdout
