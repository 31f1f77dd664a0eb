"""Every demo runs to completion on the GPU (the reference's demos/test_demos.py)."""

import pathlib
import subprocess
import sys

import pytest

from tests import helpers

pytestmark = pytest.mark.gpu
DEMOS = pathlib.Path(__file__).resolve().parent.parent / "demos"


@pytest.mark.parametrize("script,args", [
    ("demo_Y_bifurcation.py", []), ("demo_double_Y_bifurcation.py", []), ("demo_tree.py", []),
    ("demo_arterial_tree.py", []), ("demo_perf.py", ["3", "6", "12"]),
])
def test_demo(script, args, tmp_path):
    out = subprocess.run([sys.executable, str(DEMOS / script), *args], capture_output=True, text=True,
                         timeout=600, cwd=tmp_path, env={**__import__("os").environ, "PYTHONPATH": str(DEMOS.parent)})
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    if script == "demo_Y_bifurcation.py":
        assert "0.77485177" in out.stdout


@pytest.mark.parametrize("script,args", [
    ("demo_Y_bifurcation.py", []),            # too small to cut: replicated on every rank
    ("demo_arterial_tree.py", []),            # 40 cells per edge: split phases around NCCL all-reduces
    ("demo_perf.py", ["3", "8", "13"]),      # one cell per edge: in-kernel NVLink exchange
])
def test_demo_runs_unchanged_under_torchrun(script, args, tmp_path):
    """The reference's scripts run serially or under ``mpiexec -n k`` (mesh.py:84-96, CI
    test_package.yml:39-47); here the launcher is torchrun: NetworkMesh partitions the network over the
    ranks and Solver.solve() returns each rank's Functions.  Needs 2 GPUs."""
    import os

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(helpers.free_port()), str(DEMOS / script), *args]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path,
                         env={**os.environ, "PYTHONPATH": str(DEMOS.parent)})
    assert out.returncode == 0, out.stdout[-2500:] + out.stderr[-2500:]
    if script == "demo_Y_bifurcation.py":
        assert out.stdout.count("0.77485177") == 2  # both ranks solved the whole (replicated) network
