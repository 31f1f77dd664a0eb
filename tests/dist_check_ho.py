"""Multi-GPU check of higher-order elements on a partitioned network (run under torchrun):

    torchrun --nproc-per-node 2 tests/dist_check_ho.py <mode> [generations] [N] [chunk] [workload] [fd] [pd]

mode ``solver``: ``DistributedSolver(..., flux_degree=fd, pressure_degree=pd)``; ``api``: the reference-API path
(``NetworkMesh(G, N)`` cut over the ranks, ``HydraulicNetworkAssembler(nm, fd, pd)``, ``Solver(asm).solve()``);
``refuse`` (one rank): the peer exchange refuses a higher-order context, ``auto`` falls back to the all-reduces.
Workloads as in ``dist_check.py``.  ``NXFX_DIST_ONE_GPU=1``: all ranks share cuda:0 and reduce through gloo.
Rank 0 gathers the solution and compares it with the oracle's direct solve of the WHOLE network (1e-8 rel. L2)."""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import networks_fenicsx_b200 as nxfx  # noqa: E402
from networks_fenicsx_b200.distributed import DistributedSolver  # noqa: E402
from networks_fenicsx_b200.mesh import _edge_colors  # noqa: E402
from tests.dist_check import build_workload  # noqa: E402
from tests.ho_partition import expected_exchange_sizes, oracle_ho, place  # noqa: E402


def whole_network_solution(G, N, fd, pd, p_bc, R, f):
    colors = _edge_colors(G, "smallest_last", np.asarray(G.edges, dtype=np.int64))
    net = oracle_ho(G.pos, G.edges, colors, N, fd, pd)
    Rc = 1.0 if R is None else (np.repeat(R, N) if np.ndim(R) and np.size(R) == G.number_of_edges() else R)
    A, b = net.assemble(net.eval_pbc(p_bc), R=Rc, f=0.0 if f is None else f)
    return net, A, b, net.solve(A, b)


def check_sizes(ds, fd, pd):
    s, a, r = C.c_int32(0), C.c_int32(0), C.c_int32(0)
    ds.dev.call("nxfx_exchange_sizes", C.byref(s), C.byref(a), C.byref(r))
    assert (s.value, a.value, r.value) == expected_exchange_sizes(ds.part.n_top, pd >= 1), (s.value, a.value, r.value)


def run_solver(rank, world, device, exchange, n, N, chunk, workload, fd, pd):
    G, p_bc, R, f = build_workload(workload, n, N)
    ds = DistributedSolver(G, N, p_bc, R=R, f=f, device=device, chunk_nodes=chunk, exchange=exchange,
                           flux_degree=fd, pressure_degree=pd)
    assert ds.exchange == "nccl"
    check_sizes(ds, fd, pd)
    ds.assemble()
    hist = ds.solve(refine_steps=1, final_residual=True)
    if workload == "tree":
        assert ds.corrections == 0, f"the distributed direct solve needed {ds.corrections} correction(s) on a tree: {hist}"
    first = ds.dof_values()
    ds.assemble()  # a second step on the same objects
    hist2 = ds.solve(refine_steps=1, final_residual=False)
    vals = ds.dof_values()
    again = max(float(np.abs(vals[k] - first[k]).max(initial=0.0)) for k in ("flux", "pressure", "node_pressure", "lam"))
    # the replicated nodal unknowns of the shared bifurcations (exchanged order): bit-identical on every rank
    xl, sh = ds.local_solution(), ds.part.shared_lm
    rows = [xl.size - ds.part.global_bif.size + sh]
    if pd >= 1:
        rows.append(ds.part.global_edges.size * (fd * N + 1) + ds.mesh.bifurcation_values[sh])
    replicated = np.concatenate([xl[r] for r in rows])
    gathered = [None] * world
    dist.gather_object((vals, again, replicated), gathered if rank == 0 else None, dst=0)
    if rank != 0:
        return True
    assert all(np.array_equal(g[2], gathered[0][2]) for g in gathered), "replicated nodal unknowns differ between ranks"
    net, A, b, x_ref = whole_network_solution(G, N, fd, pd, p_bc, R, f)
    x = place(net, [g[0] for g in gathered])
    assert not np.isnan(x).any(), "some dofs were not owned by any rank"
    err = np.linalg.norm(x - x_ref) / np.linalg.norm(x_ref)
    res = np.linalg.norm(A @ x - b) / np.linalg.norm(b)
    drift = max(g[1] for g in gathered) / np.abs(x_ref).max()
    # the table-driven assembly matches the oracle's values to rounding, not bit for bit: the residual of the
    # device's solution against the oracle's matrix has a floor of ~1e-15 (a few e-15 with the arterial R ~ r^-4)
    floor = 1e-14
    ok = (err < 1e-8 and 0.2 * res - floor <= hist[-1] <= 5 * res + floor and drift < 1e-10
          and abs(hist2[0] - hist[0]) <= 1e-3 * hist[0] + 1e-15 and ds.n_dofs_global == net.n_dofs)
    print(f"dist_check_ho solver world={world} workload={workload} n={n} N={N} P{fd}/{'DG0' if pd == 0 else f'P{pd}'}: "
          f"dofs={net.n_dofs} (allreduce {ds.n_dofs_global}) n_top={ds.part.n_top} corrections={ds.corrections} "
          f"rel L2 error vs direct solve {err:.2e}, true residual {res:.2e}, reported residuals {hist} / {hist2}, "
          f"second step drift {drift:.1e} -> {'OK' if ok else 'FAIL'}", flush=True)
    return ok


def run_api(rank, world, device, n, N, workload, fd, pd, one_gpu):
    from networks_fenicsx_b200.parallel import TorchDistComm

    G, p_bc, _, _ = build_workload(workload, n, N)
    f = 0.5
    # the reference's script, unchanged: NetworkMesh cuts the network over the ranks of the process group
    nm = nxfx.NetworkMesh(G, N, comm=TorchDistComm() if one_gpu else None, device=device if one_gpu else None)
    assert nm._partition is not None
    asm = nxfx.HydraulicNetworkAssembler(nm, flux_degree=fd, pressure_degree=pd)
    asm.compute_forms(p_bc_ex=p_bc, f=f)
    solver = nxfx.Solver(asm)
    solver.assemble()
    fns = solver.solve()
    ds = solver._dist
    assert ds is not None and ds.exchange == "nccl"
    local = np.concatenate([fn.x.array for fn in fns])
    same = bool(np.array_equal(local, ds.local_solution()))
    gathered = [None] * world
    dist.gather_object((ds.dof_values(), same), gathered if rank == 0 else None, dst=0)
    if rank != 0:
        return True
    net, A, b, x_ref = whole_network_solution(G, N, fd, pd, p_bc, None, f)
    x = place(net, [g[0] for g in gathered])
    assert not np.isnan(x).any(), "some dofs were not owned by any rank"
    err = np.linalg.norm(x - x_ref) / np.linalg.norm(x_ref)
    ok = err < 1e-8 and all(g[1] for g in gathered) and ds.n_dofs_global == net.n_dofs
    print(f"dist_check_ho api world={world} workload={workload} n={n} N={N} P{fd}/{'DG0' if pd == 0 else f'P{pd}'}: "
          f"dofs={net.n_dofs} rel L2 error vs direct solve {err:.2e}, ksp its {solver.ksp.its} "
          f"-> {'OK' if ok else 'FAIL'}", flush=True)
    return ok


def run_refuse(device, n, N, chunk, workload, fd, pd):
    G, p_bc, R, f = build_workload(workload, n, N)
    ds = DistributedSolver(G, N, p_bc, R=R, f=f, device=device, chunk_nodes=chunk, exchange="nccl",
                           flux_degree=fd, pressure_degree=pd)
    handle, slot = (C.c_ubyte * 64)(), C.c_int32(0)
    rc = ds.dev.lib.nxfx_comm_create(ds.dev.handle, 0, 2, C.cast(handle, C.c_void_p), C.byref(slot))
    assert rc == -5, f"nxfx_comm_create on a higher-order context returned {rc}, expected NXFX_ERR_UNSUPPORTED"
    try:
        DistributedSolver(G, N, p_bc, R=R, f=f, device=device, chunk_nodes=chunk, exchange="peer",
                          flux_degree=fd, pressure_degree=pd)
        raise AssertionError("exchange='peer' accepted a higher-order context")
    except RuntimeError as exc:
        assert "flux degree 1" in str(exc), exc
    auto = DistributedSolver(G, N, p_bc, R=R, f=f, device=device, chunk_nodes=chunk, exchange="auto",
                             flux_degree=fd, pressure_degree=pd)
    assert auto.exchange == "nccl", auto.exchange
    print("dist_check_ho refuse: comm_create -> UNSUPPORTED, peer raises, auto -> nccl -> OK", flush=True)
    return True


def main():
    mode = sys.argv[1]
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 8
    N = int(sys.argv[3]) if len(sys.argv) > 3 else 2
    chunk = int(sys.argv[4]) if len(sys.argv) > 4 else 32
    workload = sys.argv[5] if len(sys.argv) > 5 else "tree"
    fd = int(sys.argv[6]) if len(sys.argv) > 6 else 2
    pd = int(sys.argv[7]) if len(sys.argv) > 7 else 1
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    one_gpu = os.environ.get("NXFX_DIST_ONE_GPU") == "1"
    if one_gpu:  # every rank on cuda:0, collectives through gloo (see dist_check.py)
        local_rank = 0
        torch.cuda.set_device(0)
        dist.init_process_group("gloo")
    else:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rank, world = dist.get_rank(), dist.get_world_size()
    if mode == "solver":
        ok = run_solver(rank, world, local_rank, "nccl" if one_gpu else "auto", n, N, chunk, workload, fd, pd)
    elif mode == "api":
        ok = run_api(rank, world, local_rank, n, N, workload, fd, pd, one_gpu)
    else:
        ok = run_refuse(local_rank, n, N, chunk, workload, fd, pd)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
