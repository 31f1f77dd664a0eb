"""One network cut into parts that are threads of ONE process (``PartitionedSolver``), against the oracle's
direct solve of the whole network -- the bars of ``tests/dist_check.py`` and ``tests/dist_check_ho.py``
without a launcher.  With ``devices=[0, 0, ...]`` the in-kernel peer exchange (``peer.cuh``: the fused
cooperative tree kernel and the last block of the residual kernel) runs between ranks on one GPU."""

import numpy as np
import pytest

import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200.mesh import _edge_colors
from networks_fenicsx_b200.schedule import build_tree_schedule
from tests.dist_check import build_workload
from tests.dist_check_ho import whole_network_solution
from tests.ho_partition import place

pytestmark = pytest.mark.gpu


def oracle_p1(G, N, p_bc, R, f):
    from oracle import reference_port as rp

    colors = _edge_colors(G, "smallest_last", np.asarray(G.edges, dtype=np.int64))
    net = rp.OracleNetwork(G.pos, G.edges, colors, N)
    Rc = 1.0 if R is None else np.repeat(R, N)
    A, b = net.assemble(net.eval_pbc(p_bc), R=Rc, f=0.0 if f is None else f)
    return net, A, b, net.solve(A, b)


def place_p1(net, N, vals):
    x = np.full(net.n_dofs, np.nan)
    for v in vals:
        ge = np.asarray(v["edges"], dtype=np.int64)
        x[net.fb[ge][:, None] + np.arange(N + 1)[None, :]] = v["flux"]
        x[net.pb[ge][:, None] + np.arange(N)[None, :]] = v["pressure"]
        x[net.loff + np.asarray(v["multipliers"], dtype=np.int64)] = v["lam"]
    return x


def single_gpu_launches(G, N, p_bc, R, f, chunk):
    """Kernel launches of one solve of the WHOLE network by ``Solver`` on one GPU, same chunk size."""
    nm = nxfx.NetworkMesh(G, N=N)
    asm = nxfx.HydraulicNetworkAssembler(nm)
    asm.compute_forms(p_bc_ex=p_bc, f=f, R=R)
    sched = build_tree_schedule(nm.graph_edges, nm.node_multiplier_index, nm.bifurcation_values.size,
                                root_hint_nodes=nm._boundary_out_nodes, chunk_nodes=chunk)
    s = nxfx.Solver(asm, schedule=sched)
    s.assemble()
    l0 = nm.device.launch_count
    s.solve()
    return nm.device.launch_count - l0


def replicated(ds, pd):
    """The replicated unknowns of the shared bifurcations: multipliers and, for a continuous pressure, nodal
    pressures."""
    xl, sh = ds.local_solution(), ds.part.shared_lm
    rows = [xl.size - ds.part.global_bif.size + sh]
    if pd >= 1:
        fd = ds.assembler.degrees[0]
        rows.append(ds.part.global_edges.size * (fd * ds.mesh.cells_per_edge + 1) + ds.mesh.bifurcation_values[sh])
    return np.concatenate([xl[r] for r in rows])


def check_partitioned(workload, n, N, chunk, exchange, devices, expect, fd=1, pd=0):
    G, p_bc, R, f = build_workload(workload, n, N)
    with nxfx.PartitionedSolver(G, N, p_bc, f=f, R=R, devices=devices, flux_degree=fd, pressure_degree=pd,
                                exchange=exchange, chunk_nodes=chunk) as ps:
        assert ps.exchange == expect
        assert ps.map(lambda s: s.exchange) == [expect] * len(devices)
        ps.assemble()
        hist = ps.solve(refine_steps=1, final_residual=True)
        assert all(h == hist for h in ps.map(lambda s: s.history)), "the residual history differs between ranks"
        if workload == "tree":
            assert ps.map(lambda s: s.corrections) == [0] * len(devices), hist
        first = ps.dof_values()
        # a second step on the same objects: the epochs and parities of the peer exchange advance
        ps.assemble()
        l0 = ps.map(lambda s: s.dev.launch_count)
        hist2 = ps.solve(refine_steps=1, final_residual=False)
        launches = [b - a for a, b in zip(l0, ps.map(lambda s: s.dev.launch_count))]
        vals = ps.dof_values()
        reps = ps.map(lambda s: replicated(s, pd))
        n_global = ps.map(lambda s: s.n_dofs_global)
    assert all(np.array_equal(r, reps[0]) for r in reps), "replicated unknowns differ between ranks"
    if (fd, pd) == (1, 0):
        net, A, b, x_ref = oracle_p1(G, N, p_bc, R, f)
        x = place_p1(net, N, vals)
        floor = 1e-17
    else:
        net, A, b, x_ref = whole_network_solution(G, N, fd, pd, p_bc, R, f)
        x = place(net, vals)
        floor = 1e-14  # the table-driven assembly matches the oracle's values to rounding (dist_check_ho.py)
    assert not np.isnan(x).any(), "some dofs were not owned by any rank"
    err = np.linalg.norm(x - x_ref) / np.linalg.norm(x_ref)
    res = np.linalg.norm(A @ x - b) / np.linalg.norm(b)
    assert err < 1e-8, err
    assert 0.2 * res - floor <= hist[-1] <= 5 * res + floor, (hist, res)  # the reported residual is the true one
    assert abs(hist2[0] - hist[0]) <= 1e-3 * hist[0] + floor, (hist, hist2)
    drift = max(float(np.abs(v[k] - w[k]).max(initial=0.0)) for v, w in zip(vals, first)
                for k in ("flux", "pressure", "node_pressure", "lam"))
    assert drift <= 1e-10 * np.abs(x_ref).max(), drift
    assert n_global == [net.n_dofs] * len(devices)
    if (fd, pd) == (1, 0) and expect == "peer":
        assert launches == [single_gpu_launches(G, N, p_bc, R, f, chunk)] * len(devices), launches
    return G


@pytest.mark.parametrize("workload,n,N,chunk,exchange", [
    ("tree", 11, 1, 64, "peer"),
    ("arterial", 10, 1, 64, "peer"),   # radius-dependent R, f != 0
    ("tree", 9, 4, 32, "auto"),        # 4 cells per edge: fused kernels with array staging
])
def test_peer_exchange_two_parts_one_gpu(workload, n, N, chunk, exchange):
    check_partitioned(workload, n, N, chunk, exchange, [0, 0], "peer")


def test_peer_exchange_four_parts_one_gpu():
    """Four cooperative grids on one device.  The tree kernel runs 1024 threads a block, so at most 2 blocks an
    SM: the grids fit together when their blocks sum to at most one per SM -- here a few blocks each."""
    import torch

    from networks_fenicsx_b200.distributed import partition_tree

    G, _, _, _ = build_workload("tree", 10, 1)
    grids = [partition_tree(G, 4, r, 32).schedule.n_chunks for r in range(4)]  # bottom chunks + the top block
    assert sum(grids) <= torch.cuda.get_device_properties(0).multi_processor_count
    check_partitioned("tree", 10, 1, 32, "peer", [0, 0, 0, 0], "peer")


@pytest.mark.parametrize("fd,pd,N", [(2, 1, 2), (2, 0, 3), (2, 1, 3)])
def test_higher_order_split_phases_one_gpu(fd, pd, N):
    check_partitioned("tree", 8, N, 32, "auto", [0, 0], "nccl", fd=fd, pd=pd)


def test_grids_that_cannot_be_resident_together():
    """Chunks of 4 nodes: each rank's cooperative tree grid has more blocks than there are SMs, so two of them
    exceed the 2 blocks an SM of the 1024-thread tree kernel.  ``peer`` is refused before any launch and names
    the limit; ``auto`` falls back to the split phases and solves."""
    import torch

    from networks_fenicsx_b200.distributed import partition_tree

    G, p_bc, _, _ = build_workload("tree", 12, 1)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert all(partition_tree(G, 2, r, 4).schedule.n_chunks > sms for r in range(2))
    with pytest.raises(RuntimeError, match="not resident together"):
        nxfx.PartitionedSolver(G, 1, p_bc, devices=[0, 0], exchange="peer", chunk_nodes=4)
    with nxfx.PartitionedSolver(G, 1, p_bc, devices=[0, 0], exchange="nccl", chunk_nodes=4) as ref:
        built = ref.map(lambda s: s.dev.launch_count)
    with nxfx.PartitionedSolver(G, 1, p_bc, devices=[0, 0], exchange="auto", chunk_nodes=4) as ps:
        assert ps.exchange == "nccl"
        assert ps.map(lambda s: s.dev.launch_count) == built  # the refused connection launched nothing
    check_partitioned("tree", 12, 1, 4, "auto", [0, 0], "nccl")


@pytest.mark.parametrize("fd,pd,exchange,expect", [(1, 0, "peer", "peer"), (2, 1, "auto", "nccl")])
def test_two_gpus_in_one_process(fd, pd, exchange, expect):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    if (fd, pd) == (1, 0):
        check_partitioned("tree", 11, 1, 64, exchange, [0, 1], expect)
    else:
        check_partitioned("tree", 8, 2, 32, exchange, [0, 1], expect, fd=fd, pd=pd)
