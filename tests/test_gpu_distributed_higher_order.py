"""Higher-order elements on a network cut over several ranks (tests/dist_check_ho.py under torchrun): the gathered
solution against the oracle's direct solve of the whole network, through DistributedSolver and through the
reference API (NetworkMesh + HydraulicNetworkAssembler + Solver), and the refusal of the in-kernel peer exchange.
The one-GPU cases run every rank on cuda:0 with gloo collectives (host-driven exchange); the 2-GPU cases use NCCL
on separate devices and are skipped below 2 GPUs."""

import os
import pathlib
import subprocess
import sys

import pytest

from tests import helpers

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parent.parent

SOLVER_CASES = [
    (("solver", "8", "2", "32", "tree", "2", "1"), 2),      # P2/P1 tree
    (("solver", "6", "2", "16", "arterial", "3", "2"), 2),  # P3/P2, radius-dependent R, f != 0
    (("solver", "8", "3", "16", "tree", "2", "0"), 4),      # P2/DG0
    (("solver", "7", "2", "16", "arterial", "2", "1"), 3),  # P2/P1 arterial, odd world
]
API_CASE = (("api", "8", "2", "0", "tree", "2", "1"), 2)


def torchrun(args, world, one_gpu, timeout=600):
    env = dict(os.environ)
    if one_gpu:
        env["NXFX_DIST_ONE_GPU"] = "1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(helpers.free_port()),
           str(ROOT / "tests" / "dist_check_ho.py"), *args]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "-> OK" in out.stdout, out.stdout[-3000:]


@pytest.mark.parametrize("args,world", [*SOLVER_CASES, API_CASE])
def test_higher_order_partition_ranks_sharing_one_gpu(args, world):
    torchrun(args, world, one_gpu=True)


def test_peer_exchange_refuses_higher_order():
    """nxfx_comm_create returns NXFX_ERR_UNSUPPORTED on a higher-order context, exchange='peer' raises and
    exchange='auto' falls back to the host-driven all-reduces."""
    torchrun(("refuse", "8", "2", "32", "tree", "2", "1"), 1, one_gpu=True)


@pytest.mark.parametrize("args,world", [SOLVER_CASES[0], SOLVER_CASES[1], API_CASE])
def test_higher_order_partition_two_gpus(args, world):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    torchrun(args, world, one_gpu=False)
