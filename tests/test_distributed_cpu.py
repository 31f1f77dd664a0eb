"""world_size-2 gloo test (CPU) of the multi-GPU host path: component partition of a forest,
local sub-networks, and the metadata collectives.  No GPU compute."""

import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200 import network_generation as ng
from networks_fenicsx_b200 import parallel
from tests import helpers


def make_forest():
    trees = [ng.make_tree(n, n, n, as_arrays=True) for n in (6, 4, 5, 6)]
    for k, t in enumerate(trees):
        t.pos[:, 0] += 100.0 * k
    return parallel.forest(trees)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        F = make_forest()
        rank_of_edge = parallel.partition_components(F.edges, F.number_of_nodes(), world)
        part = parallel.local_part(F, rank_of_edge, rank)
        nm = nxfx.NetworkMesh(part.graph, N=3, color_strategy="smallest_last")
        asm = nxfx.HydraulicNetworkAssembler(nm)
        comm = parallel.TorchDistComm()
        total_dofs = comm.allreduce(asm.num_dofs)
        total_edges = comm.allreduce(part.global_edges.size)
        max_edges = comm.allreduce(part.global_edges.size, op=max)
        meta = comm.bcast({"dofs": asm.num_dofs} if rank == 0 else None, root=0)
        comm.barrier()
        out[rank] = (asm.num_dofs, part.n_components, total_dofs, total_edges, max_edges, meta["dofs"],
                     int(nm.bifurcation_values.size), part.global_nodes.tolist() == sorted(part.global_nodes.tolist()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_forest_partition_world2():
    world = 2
    with mp.Manager() as manager:
        out = manager.dict()
        mp.spawn(_worker, args=(world, helpers.free_port(), out), nprocs=world, join=True)
        res = dict(out)
    F = make_forest()
    whole = nxfx.HydraulicNetworkAssembler(nxfx.NetworkMesh(F, N=3, color_strategy="smallest_last"))
    assert sum(r[0] for r in res.values()) == whole.num_dofs == int(res[0][2])
    assert sum(r[1] for r in res.values()) == 4
    assert int(res[0][3]) == F.number_of_edges()
    # LPT packing of trees with 63, 15, 31, 63 edges: {63, 31} and {63, 15}
    assert int(res[0][4]) == 94
    assert res[1][5] == res[0][0]
    assert all(r[7] for r in res.values())


def test_partition_is_deterministic_and_balanced():
    F = make_forest()
    r1 = parallel.partition_components(F.edges, F.number_of_nodes(), 4)
    r2 = parallel.partition_components(F.edges, F.number_of_nodes(), 4)
    assert np.array_equal(r1, r2)
    assert sorted(np.bincount(r1).tolist()) == [15, 31, 63, 63]
    part = parallel.local_part(F, r1, int(r1[0]))
    assert part.n_components == 1 and part.graph.number_of_edges() == 63
    np.testing.assert_array_equal(F.pos[part.global_nodes], part.graph.pos)
    np.testing.assert_array_equal(part.global_nodes[part.graph.edges], F.edges[part.global_edges])
