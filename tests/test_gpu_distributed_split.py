"""The split phases of the partitioned preconditioner on their own (tests/dist_check_split.py under torchrun, both
ranks on cuda:0 with gloo collectives): setup and application through the four separate begin/end calls against
the fused setup+apply pair, and a forced refinement correction (apply_end with add = 1) against the oracle's
direct solve of the whole network."""

import pathlib
import subprocess
import sys

import pytest

from tests import helpers

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("args", [
    ("11", "1", "64", "tree", "1", "0"),     # P1/DG0, one cell per edge (fused bottom kernels of its own)
    ("8", "4", "32", "arterial", "1", "0"),  # P1/DG0, 4 cells per edge, radius-dependent R, f != 0
    ("8", "2", "32", "tree", "2", "1"),      # P2/P1
    ("8", "3", "16", "tree", "2", "0"),      # P2/DG0
])
def test_split_phases_ranks_sharing_one_gpu(args):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(helpers.free_port()),
           str(ROOT / "tests" / "dist_check_split.py"), *args]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "-> OK" in out.stdout, out.stdout[-3000:]
    print(out.stdout.strip().splitlines()[-1])
