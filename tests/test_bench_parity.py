"""bench.py's host-side parity checks (matrix-free residual, Kirchhoff sums, Thevenin closed form),
validated on the CPU against the oracle's direct solve: a correct solution passes, a perturbed one fails."""

import pathlib
import subprocess
import sys
import types

import numpy as np
import pytest

import bench
import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200 import network_generation as ng
from oracle import reference_port as rp


def fake_problem(G, N, R_edge, f_cell, x, nm, net):
    asm = types.SimpleNamespace(_pbc_host=net.eval_pbc(bench.p_bc))
    solver = types.SimpleNamespace(x=types.SimpleNamespace(array_r=x))
    nm._x_host = net.x3  # stands in for the device-generated vertices
    return types.SimpleNamespace(nm=nm, asm=asm, solver=solver, N=N, ds=None, G=G, R_edge=R_edge, f_cell=f_cell)


@pytest.mark.parametrize("workload,n,N", [("tree", 7, 1), ("tree", 5, 3), ("arterial", 6, 1), ("arterial", 5, 4)])
def test_host_parity_accepts_the_direct_solution_and_rejects_a_wrong_one(workload, n, N):
    G, R, f = bench.make_workload(workload, n, N)
    nm = nxfx.NetworkMesh(G, N=N, color_strategy="smallest_last")
    net = rp.OracleNetwork(G.pos, G.edges, nm.edge_colors, N)
    A, b = net.assemble(net.eval_pbc(bench.p_bc), R=1.0 if R is None else np.repeat(R, N), f=0.0 if f is None else f)
    x = net.solve(A, b)
    par = bench.host_parity(fake_problem(G, N, R, f, x, nm, net), None, None)
    true_res = np.linalg.norm(A @ x - b) / np.linalg.norm(b)
    assert par["true_residual_recomputed"] < 1e-12 and abs(par["true_residual_recomputed"] - true_res) < 1e-13
    assert par["kirchhoff_max"] < 1e-12
    if f is None:
        assert par["q_const_max"] < 1e-10
        assert par["rel_l2_vs_closed_form"]["flux"] < 1e-10 and par["rel_l2_vs_closed_form"]["multipliers"] < 1e-10
    else:
        assert par["rel_l2_vs_closed_form"] is None
    bad = x.copy()
    bad[net.loff + 1] += 1e-3
    par_bad = bench.host_parity(fake_problem(G, N, R, f, bad, nm, net), None, None)
    assert par_bad["true_residual_recomputed"] > 1e-6
    if f is None:
        assert par_bad["rel_l2_vs_closed_form"]["multipliers"] > 1e-6


def test_closed_form_with_radius_dependent_resistance():
    """f = 0 with R_e = 8 mu / (pi r^4): the Thevenin reduction equals the oracle's resistor-network solve."""
    G, R, _ = bench.make_workload("arterial", 7, 1)
    nm = nxfx.NetworkMesh(G, N=2, color_strategy="smallest_last")
    net = rp.OracleNetwork(G.pos, G.edges, nm.edge_colors, 2)
    A, b = net.assemble(net.eval_pbc(bench.p_bc), R=np.repeat(R, 2))
    x = net.solve(A, b)
    par = bench.host_parity(fake_problem(G, 2, R, None, x, nm, net), None, None)
    assert par["rel_l2_vs_closed_form"]["flux"] < 1e-9 and par["rel_l2_vs_closed_form"]["multipliers"] < 1e-9
    q_edge, lam = net.resistor_network_solution(net.eval_pbc(bench.p_bc), R=np.repeat(R, 2))
    assert np.allclose(x[net.loff:], lam, rtol=1e-9, atol=1e-12)


def test_dump_outputs_writes_float64_and_samples_above_the_cap(tmp_path):
    small = {"a": np.arange(10, dtype=np.float32), "b": np.linspace(0.0, 1.0, 7)}
    bench.dump_outputs(tmp_path / "all", small)
    for name, a in small.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, a)
    big = {"x": np.arange(40000, dtype=np.float64), "y": -np.arange(20000, dtype=np.float64)}
    cap = 100_000
    for d in ("s1", "s2"):
        bench.dump_outputs(tmp_path / d, big, max_bytes=cap)
    assert sum(f.stat().st_size for f in (tmp_path / "s1").iterdir()) <= cap
    for name, a in big.items():
        s1, s2 = np.load(tmp_path / "s1" / f"{name}.npy"), np.load(tmp_path / "s2" / f"{name}.npy")
        assert np.array_equal(s1, s2), "the sample differs between two runs"
        assert 0 < s1.size < a.size and np.all(np.isin(s1, a)) and np.all(np.diff(np.abs(s1)) > 0)


@pytest.mark.gpu
def test_bench_dumps_the_solution_of_the_timed_step(tmp_path):
    """``bench.py --dump-outputs``: the blocks of the last timed step are the oracle's direct solve."""
    n = 8
    cmd = [sys.executable, str(pathlib.Path(bench.__file__)), "--generations", str(n), "--steps", "2", "--warmup", "1",
           "--strong-generations", "0", "--higher-order-generations", "0", "--no-cpu-baseline",
           "--dump-outputs", str(tmp_path / "out")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    G, _, _ = bench.make_workload("tree", n, 1)
    nm = nxfx.NetworkMesh(G, N=1, color_strategy="smallest_last")
    net = rp.OracleNetwork(G.pos, G.edges, nm.edge_colors, 1)
    A, b = net.assemble(net.eval_pbc(bench.p_bc))
    x_ref = net.solve(A, b)
    C = int(nm.edge_colors.max()) + 1
    names = [f"flux_color_{i}" for i in range(C)] + ["pressure", "global_flux"]
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == sorted(f"{k}.npy" for k in names)
    blocks = [np.load(tmp_path / "out" / f"{k}.npy") for k in names]
    assert all(blk.dtype == np.float64 for blk in blocks)
    x = np.concatenate(blocks)
    assert x.size == x_ref.size and np.linalg.norm(x - x_ref) / np.linalg.norm(x_ref) < 1e-10
