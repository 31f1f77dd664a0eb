"""Split phases of the partitioned preconditioner, called one by one (run under torchrun; every rank on cuda:0,
collectives through gloo, so a single-GPU box runs it):

    torchrun --nproc-per-node 2 tests/dist_check_split.py [generations] [N] [chunk] [workload] [fd] [pd]

* unfused vs fused: ``nxfx_pc_setup_begin`` -> all-reduce -> ``_setup_end``, then ``nxfx_pc_apply_begin`` ->
  all-reduce -> ``_apply_end`` (add = 0) gives the z of ``nxfx_pc_setup_apply_begin`` -> all-reduce ->
  ``_setup_apply_end``.  Bit-identical where the fused call is that composition; P1/DG0 with one cell per edge
  has fused bottom kernels of its own and is compared to 1e-13 (relative, max norm).
* forced correction: ``DistributedSolver.solve(refine_steps=1, refine_rtol=0)`` applies one correction
  (``_apply_end`` with add = 1); the gathered solution matches the oracle's direct solve of the whole network
  (1e-8 rel. L2) and the reported residual the true one.
Workloads as in ``dist_check.py``."""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from networks_fenicsx_b200.distributed import DistributedSolver  # noqa: E402
from tests.dist_check import build_workload  # noqa: E402
from tests.dist_check_ho import whole_network_solution  # noqa: E402
from tests.ho_partition import place  # noqa: E402


def preconditioner(ds, fused):
    """z = P^{-1} b through the split phases, with the caller's all-reduces in between."""
    dev = ds.dev
    ns, na = C.c_int32(0), C.c_int32(0)
    dev.call("nxfx_exchange_sizes", C.byref(ns), C.byref(na), C.byref(C.c_int32(0)))
    ns, na = ns.value, na.value
    top = torch.zeros(ns + na, dtype=torch.float64, device="cuda:0")
    z = torch.zeros(ds.assembler.num_dofs, dtype=torch.float64, device="cuda:0")

    def ptr(t, offset=0):
        return C.c_void_p(t.data_ptr() + 8 * offset)

    b = ds.solver.b.device_ptr()
    if fused:
        dev.call("nxfx_pc_setup_apply_begin", b, ptr(top))
        dist.all_reduce(top)
        dev.call("nxfx_pc_setup_apply_end", b, ptr(z), ptr(top))
    else:
        dev.call("nxfx_pc_setup_begin", ptr(top))
        dist.all_reduce(top[:ns])
        dev.call("nxfx_pc_setup_end", ptr(top))
        dev.call("nxfx_pc_apply_begin", b, ptr(top, ns))
        dist.all_reduce(top[ns:])
        dev.call("nxfx_pc_apply_end", b, ptr(z), ptr(top, ns), 0)
    dev.sync()
    return z.cpu().numpy()


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    N = int(sys.argv[2]) if len(sys.argv) > 2 else 1
    chunk = int(sys.argv[3]) if len(sys.argv) > 3 else 32
    workload = sys.argv[4] if len(sys.argv) > 4 else "tree"
    fd = int(sys.argv[5]) if len(sys.argv) > 5 else 1
    pd = int(sys.argv[6]) if len(sys.argv) > 6 else 0
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    G, p_bc, R, f = build_workload(workload, n, N)
    ds = DistributedSolver(G, N, p_bc, R=R, f=f, device=0, chunk_nodes=chunk, exchange="nccl",
                           flux_degree=fd, pressure_degree=pd)
    ds.assemble()
    z_split = preconditioner(ds, fused=False)
    z_fused = preconditioner(ds, fused=True)
    same = bool(np.array_equal(z_split, z_fused))
    diff = float(np.abs(z_split - z_fused).max() / np.abs(z_fused).max())
    hist = ds.solve(refine_steps=1, refine_rtol=0.0, final_residual=True)
    gathered = [None] * world
    dist.gather_object((ds.dof_values(), same, diff, ds.corrections), gathered if rank == 0 else None, dst=0)
    ok = True
    if rank == 0:
        net, A, b, x_ref = whole_network_solution(G, N, fd, pd, p_bc, R, f)
        x = place(net, [g[0] for g in gathered])
        assert not np.isnan(x).any(), "some dofs were not owned by any rank"
        err = np.linalg.norm(x - x_ref) / np.linalg.norm(x_ref)
        res = np.linalg.norm(A @ x - b) / np.linalg.norm(b)
        # only P1/DG0 with one cell per edge has fused kernels of its own; elsewhere the fused call IS the composition
        own_kernels = fd == 1 and pd == 0 and N == 1
        bit = all(g[1] for g in gathered)
        worst = max(g[2] for g in gathered)
        floor = 1e-14  # the residual against the oracle's matrix has a rounding floor (see dist_check_ho.py)
        ok = ((bit or (own_kernels and worst <= 1e-13)) and all(g[3] == 1 for g in gathered) and err < 1e-8
              and 0.2 * res - floor <= hist[-1] <= 5 * res + floor)
        print(f"dist_check_split world={world} workload={workload} n={n} N={N} P{fd}/{'DG0' if pd == 0 else f'P{pd}'}: "
              f"unfused vs fused z bit-identical={bit} (max rel diff {worst:.1e}), corrections="
              f"{[g[3] for g in gathered]}, rel L2 error vs direct solve {err:.2e}, true residual {res:.2e}, "
              f"reported residuals {hist} -> {'OK' if ok else 'FAIL'}", flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
