"""Device functions on a partitioned network (run under torchrun, every rank on cuda:0, gloo collectives):

    NXFX_DIST_ONE_GPU=1 torchrun --nproc-per-node 2 tests/dist_check_device.py [generations] [N] [fd] [pd]

The reference-API path (``NetworkMesh(G, N, comm=TorchDistComm())`` cut over the ranks, ``Solver(asm)``, whose
solve goes through the distributed layer) with higher-order elements, so that the exchange is the host-driven one
that ranks sharing a GPU can run.  ``R`` is given as a CUDA tensor of the whole network (restricted on the device).
Every rank checks that ``solve(create_functions(device=True))`` holds exactly the local dofs that ``solve()``
returns and that ``export_functions`` writes the same files for both."""
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import networks_fenicsx_b200 as nxfx  # noqa: E402
from networks_fenicsx_b200.parallel import TorchDistComm  # noqa: E402


def check(n, N, fd, pd):
    G = nxfx.network_generation.make_tree(n, n, n, as_arrays=True)
    E = G.number_of_edges()
    R = np.linspace(0.5, 2.0, E)
    nm = nxfx.NetworkMesh(G, N, comm=TorchDistComm(), device=0)
    assert nm._partition is not None
    asm = nxfx.HydraulicNetworkAssembler(nm, flux_degree=fd, pressure_degree=pd)
    asm.compute_forms(p_bc_ex=lambda x: x[1], R=R, f=0.5)
    solver = nxfx.Solver(asm)
    assert solver._dist is not None and solver._dist.exchange == "nccl"
    solver.assemble()
    host = solver.solve()
    x_host = np.concatenate([fn.x.array for fn in host])
    asm.compute_forms(p_bc_ex=lambda x: x[1], R=torch.from_numpy(R).cuda(), f=0.5)
    solver.assemble()
    fns = solver.solve(solver.create_functions(device=True))
    x_dev = torch.cat([fn.x.array for fn in fns]).cpu().numpy()
    same = np.array_equal(x_dev, x_host) and np.array_equal(x_dev, solver._dist.local_solution())
    with tempfile.TemporaryDirectory() as tmp:
        nxfx.post_processing.export_functions(host, os.path.join(tmp, "host"))
        nxfx.post_processing.export_functions(fns, os.path.join(tmp, "dev"))
        names = sorted(os.listdir(os.path.join(tmp, "host")))
        exported = names == sorted(os.listdir(os.path.join(tmp, "dev"))) and all(
            np.array_equal(np.load(os.path.join(tmp, "host", k)), np.load(os.path.join(tmp, "dev", k))) for k in names)
    return bool(same and exported), x_dev.size


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    N = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    fd = int(sys.argv[3]) if len(sys.argv) > 3 else 2
    pd = int(sys.argv[4]) if len(sys.argv) > 4 else 1
    assert os.environ.get("NXFX_DIST_ONE_GPU") == "1", "this check runs every rank on cuda:0"
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    ok, n_local = check(n, N, fd, pd)
    flags = torch.tensor([float(ok)])
    dist.all_reduce(flags)
    all_ok = int(flags.item()) == world
    if rank == 0:
        print(f"dist_check_device world={world} make_tree({n}) N={N} P{fd}/{'DG0' if pd == 0 else f'P{pd}'}: "
              f"device functions == solve() on every rank ({n_local} local dofs on rank 0) "
              f"-> {'OK' if all_ok else 'FAIL'}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if all_ok else 1)


if __name__ == "__main__":
    main()
