#!/usr/bin/env python
"""Benchmark of the hydraulic-network assemble+solve hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--generations n]
                    [--workload tree|arterial] [--scaling weak|strong] [--strong-generations m]
                    [--dump-outputs DIR]

A "step" is one numeric assembly (matrix + rhs) followed by one solve.  Workloads:

* ``tree`` (headline, BASELINE configs[4]): ``make_tree(n, H=n, W=n)``, ``N=1`` cell per edge,
  ``smallest_last`` colouring, flux P1 / pressure DG0, ``p_bc = y`` (demos/demo_perf.py:79-82,107,34-35)
  with n = 20 generations (3,670,012 DOFs);
* ``arterial`` (BASELINE configs[3]): ``make_arterial_tree(n)`` (demos/demo_arterial_tree.py:16-27) with
  the radius-dependent resistance ``R_e = 8 mu / (pi r_e^4)`` and a source ``f != 0``.

``value`` = DOFs / (t_assemble + t_solve) with everything resident in HBM; ``e2e`` = the same through
the Python API with host buffers (p_bc uploaded, solution downloaded every step).  With N > 1 ranks ONE
network is cut over the GPUs (weak: n + log2 N generations, strong: the same n).  Every line carries
``parity`` (size-independent checks of the returned solution, recomputed on the host in NumPy outside
the timed region), ``setup_ms`` and a ``strong`` block (the same fixed tree at every N).  Prints ONE JSON
line on rank 0.

``--dump-outputs DIR`` (single GPU) writes the solution of the last timed step as ``Solver.solve()`` hands it
out, one float64 ``DIR/<name>.npy`` per block (``flux_color_i``, ``pressure``, ``global_flux``).  The inputs
depend on the arguments only, so two builds run with the same arguments can be compared block by block.
Above 64 MB in all, every block is cut to the same share of its entries at indices drawn by a fixed seed.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tree-network assemble+solve DOFs/s"
UNIT = "DOFs/s"
MU = 1.0  # viscosity of the arterial workload


def p_bc(x):
    return x[1]


def workload_name(workload, n, N=1):
    if workload == "arterial":
        return (f"arterial tree make_arterial_tree(N={n}, direction=[0.1,1,0]), {N} cell(s)/edge, smallest_last, P1/DG0, "
                f"p_bc=y, R_e=8mu/(pi r_e^4), f=1e-3 sin(cell)")
    return f"demo_perf binary tree make_tree(n={n},H={n},W={n}), N={N}, smallest_last, P1/DG0, p_bc=y"


def make_workload(workload, n, N):
    """(graph, R per graph edge or None, f per cell or None) of the GLOBAL network."""
    from networks_fenicsx_b200 import network_generation as ng

    if workload == "arterial":
        G = ng.make_arterial_tree(N=n, direction=np.array([0.1, 1.0, 0.0]), as_arrays=True)
        radius = np.asarray(G.edge_attrs["radius"], dtype=np.float64)
        R = 8.0 * MU / (np.pi * radius**4)
        f = 1e-3 * np.sin(np.arange(G.number_of_edges() * N, dtype=np.float64))
        return G, R, f
    return ng.make_tree(n, n, n, as_arrays=True), None, None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        # nvidia-smi loops on its own and writes to a file that is parsed afterwards: no reader thread competes with
        # the timed loop for the interpreter lock (a stalled rank stalls every rank at the next exchange point)
        import tempfile

        try:
            self.out = tempfile.TemporaryFile(mode="w+")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=self.out, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.out.seek(0)
        self.lines = [ln.strip() for ln in self.out.read().splitlines()]
        self.out.close()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class Problem:
    """One workload on this rank: the single-GPU objects or this rank's part of the partitioned
    network, with the wall time of every setup phase."""

    def __init__(self, workload, n, N, device_index, world, dist):
        import networks_fenicsx_b200 as nxfx

        self.workload, self.n, self.N, self.world = workload, n, N, world
        self.setup_ms = {}
        t0 = time.perf_counter()
        self.G, self.R_edge, self.f_cell = make_workload(workload, n, N)
        self.setup_ms["generate_graph"] = (time.perf_counter() - t0) * 1e3
        self.ds = None
        if world > 1:
            from networks_fenicsx_b200.distributed import DistributedSolver

            t0 = time.perf_counter()
            self.ds = DistributedSolver(self.G, N, p_bc, R=self.R_edge, f=self.f_cell, device=device_index)
            self.setup_ms["partition_mesh_symbolic_schedule_connect"] = (time.perf_counter() - t0) * 1e3
            self.nm, self.asm, self.solver = self.ds.mesh, self.ds.assembler, self.ds.solver
            self.n_dofs_total = self.ds.n_dofs_global
            self.exchange = self.ds.exchange
        else:
            t0 = time.perf_counter()
            self.nm = nxfx.NetworkMesh(self.G, N=N, color_strategy="smallest_last", device=device_index)
            self.setup_ms["mesh_host_analysis_coloring"] = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            self.asm = nxfx.HydraulicNetworkAssembler(self.nm, flux_degree=1, pressure_degree=0)
            self.asm.compute_forms(p_bc_ex=p_bc, R=self.R_edge, f=self.f_cell)
            self.nm.device.sync()
            self.setup_ms["mesh_device_forms"] = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            self.solver = nxfx.Solver(self.asm)
            self.nm.device.sync()
            self.setup_ms["symbolic_schedule"] = (time.perf_counter() - t0) * 1e3
            self.n_dofs_total = self.asm.num_dofs
            self.exchange = "single GPU"
        self.dev = self.nm.device
        self.functions = None
        self.opts = self.solver.solve_options()
        from networks_fenicsx_b200 import _lib

        self.info = _lib.SolveInfo()
        self._lib = _lib

    def step(self):
        import ctypes as C

        if self.ds is not None:
            self.ds.assemble()
            self.ds.solve()
            return
        self.solver.assemble()
        self.dev.call("nxfx_solve", self.solver.b.device_ptr(), self.solver.x.device_ptr_overwrite(),
                      C.byref(self.opts), C.byref(self.info))

    def timed_steps(self, steps, warmup, barrier, dist, torch):
        import gc

        for _ in range(warmup):
            self.step()
        barrier()
        gc.collect()
        gc.disable()  # a collection pause on one rank stalls every rank at the next exchange point
        try:
            l0 = self.dev.launch_count
            self.dev.timer_start()
            for _ in range(steps):
                self.step()
            ms = self.dev.timer_stop()
            launches = self.dev.launch_count - l0
        finally:
            gc.enable()
        barrier()
        if dist is not None:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, launches


def colouring_note(E, world):
    """Which colouring the flux-block layout of this run comes from (mesh.color_graph)."""
    from networks_fenicsx_b200 import mesh as _mesh

    scope = "" if world == 1 else " of this rank's sub-network"
    if E <= _mesh.NETWORKX_COLORING_MAX_EDGES:
        return f"networkx greedy_color(line_graph, smallest_last){scope}: the reference's own call"
    if E <= _mesh.NETWORKX_IDENTICAL_MAX_EDGES:
        return (f"networkx-identical smallest_last{scope}, reproduced edge by edge without networkx graphs "
                "(pinned by networkx fixtures at 16 and 20 generations)")
    return f"native greedy in input order{scope} (beyond the size the networkx assignment is reproduced for; warned)"


def per_cell(coef, E, N, default):
    """Scalar / per-graph-edge / per-cell coefficient -> [E, N]."""
    if coef is None:
        return np.full((E, N), float(default))
    a = np.asarray(coef, dtype=np.float64)
    if a.ndim == 0:
        return np.full((E, N), float(a))
    if a.size == E * N:
        return a.reshape(E, N)
    if a.size == E:
        return a.reshape(E, 1) * np.ones((1, N))
    raise ValueError("coefficient must be a scalar, one value per graph edge or one per cell")


# ---- parity: size-independent checks recomputed on the host ------------------------------------------
def host_parity(pb, dist, torch):
    """Checks of the RETURNED solution that do not need an element-wise oracle and hold at any size
    (tests/test_gpu_parity.py::test_full_size_properties in bench form), recomputed in NumPy from the
    downloaded solution, the downloaded mesh vertices and the input coefficients -- independent of the
    device matrix and of the device residual.  Distributed: every rank checks its own rows; the rows of
    the replicated multipliers are summed over the ranks by one all-reduce (outside the timed region)."""
    nm, asm, N = pb.nm, pb.asm, pb.N
    x = pb.solver.x.array_r
    edges = np.asarray(nm.graph_edges)
    E = edges.shape[0]
    u, v = edges[:, 0], edges[:, 1]
    lm = np.asarray(nm.node_multiplier_index)
    fb = nm.edge_slot.astype(np.int64) * (N + 1)
    nq, nc = E * (N + 1), E * N
    q = x[fb[:, None] + np.arange(N + 1)[None, :]]  # [E, N+1]
    p = x[nq:nq + nc].reshape(E, N)
    lam = x[nq + nc:]
    X = nm.mesh.geometry.x  # device-generated vertices
    cells = nm._cells()
    d = X[cells[:, 1]] - X[cells[:, 0]]
    h = np.sqrt((d * d).sum(axis=1)).reshape(E, N)
    if pb.ds is not None:
        R = pb.ds._restrict(pb.R_edge, N, pb.G)
        f = pb.ds._restrict(pb.f_cell, N, pb.G)
    else:
        R, f = pb.R_edge, pb.f_cell
    Rc = per_cell(R, E, N, 1.0)
    fc = per_cell(f, E, N, 0.0)
    m = Rc * h
    pbc = asm._pbc_host
    lu, lv = lm[u], lm[v]
    lam_u = np.where(lu >= 0, lam[np.maximum(lu, 0)] if lam.size else 0.0, 0.0)
    lam_v = np.where(lv >= 0, lam[np.maximum(lv, 0)] if lam.size else 0.0, 0.0)
    # flux rows (assembly.py:253-255,258-260,273,277)
    Aq = np.zeros_like(q)
    Aq[:, :-1] += m / 3.0 * q[:, :-1] + m / 6.0 * q[:, 1:] + p
    Aq[:, 1:] += m / 6.0 * q[:, :-1] + m / 3.0 * q[:, 1:] - p
    Aq[:, 0] -= lam_u
    Aq[:, -1] += lam_v
    bq = np.zeros_like(q)
    bq[:, 0] = np.where(lu < 0, -pbc[u], 0.0)
    bq[:, -1] = np.where(lv < 0, pbc[v], 0.0)
    rq = bq - Aq
    # pressure rows (assembly.py:254,262)
    bp = fc * h
    rp = bp - (q[:, 1:] - q[:, :-1])
    # multiplier rows (assembly.py:272,276): sum of in-fluxes minus sum of out-fluxes = 0
    n_bif_g = pb.ds.part.n_global_bif if pb.ds is not None else lam.size
    gb = pb.ds.part.global_bif if pb.ds is not None else np.arange(lam.size)
    K = np.zeros(n_bif_g)
    np.add.at(K, gb[lv[lv >= 0]], q[lv >= 0, -1])
    np.add.at(K, gb[lu[lu >= 0]], -q[lu >= 0, 0])
    sums = np.array([float((rq * rq).sum() + (rp * rp).sum()), float((bq * bq).sum() + (bp * bp).sum())])
    qmax = float(np.abs(q).max())
    qdev = float(np.abs(q - q[:, :1]).max()) if f is None else 0.0
    if dist is not None:
        tK = torch.from_numpy(K).cuda()
        dist.all_reduce(tK)
        K = tK.cpu().numpy()
        ts = torch.from_numpy(sums).cuda()
        dist.all_reduce(ts)
        sums = ts.cpu().numpy()
        tm = torch.tensor([qmax, qdev], dtype=torch.float64, device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        qmax, qdev = (float(t) for t in tm.cpu().numpy())
    out = {
        "true_residual_recomputed": float(np.sqrt(sums[0] + float((K * K).sum())) / np.sqrt(sums[1])),
        "kirchhoff_max": float(np.abs(K).max()) if K.size else 0.0,
        "q_const_max": (qdev / qmax if qmax > 0 else 0.0) if f is None else None,
        "how": "NumPy on the host from the downloaded solution / vertices and the input coefficients (matrix-free operator "
               "of assembly.py:253-277), all rows of all ranks; closed form = Thevenin reduction of the resistor network",
    }
    out["rel_l2_vs_closed_form"] = closed_form_check(pb, q[:, 0], lam, dist, torch) if f is None else None
    return out


def closed_form_check(pb, q0_local, lam_local, dist, torch):
    """f = 0 on a rooted tree: the fluxes / multipliers are those of a resistor network with node
    potentials lambda and boundary potentials -p_bc (SURVEY A.3).  Solved on rank 0 by a leaf -> root
    Thevenin reduction (series / parallel conductances, NumPy, level by level) -- a different algorithm
    from the device's Schur elimination -- and compared with the gathered device solution."""
    G, N = pb.G, pb.N
    edges = np.asarray(G.edges, dtype=np.int64)
    E = edges.shape[0]
    n_nodes = G.number_of_nodes()
    # gather q0 per GLOBAL edge and lambda per GLOBAL multiplier (every entry has one owner)
    if pb.ds is not None:
        part = pb.ds.part
        qg = np.zeros(E)
        qg[part.global_edges] = q0_local
        lg = np.zeros(part.n_global_bif)
        own = part.lam_weight > 0
        lg[part.global_bif[own]] = lam_local[own]
        tq, tl = torch.from_numpy(qg).cuda(), torch.from_numpy(lg).cuda()
        dist.all_reduce(tq)
        dist.all_reduce(tl)
        qg, lg = tq.cpu().numpy(), tl.cpu().numpy()
        if dist.get_rank() != 0:
            return None
    else:
        qg, lg = q0_local, lam_local
    u, v = edges[:, 0], edges[:, 1]
    pos = np.asarray(G.pos, dtype=np.float64)
    length = np.sqrt(((pos[v] - pos[u]) ** 2).sum(axis=1))
    R = np.ones(E) if pb.R_edge is None else np.asarray(pb.R_edge, dtype=np.float64)
    g = 1.0 / (R * length)  # N equal cells of R h each
    deg = np.bincount(u, minlength=n_nodes) + np.bincount(v, minlength=n_nodes)
    indeg = np.bincount(v, minlength=n_nodes)
    if indeg.max() > 1 or (indeg == 0).sum() != 1 or deg[np.flatnonzero(indeg == 0)[0]] != 1:
        return None  # not an out-tree hanging below a single inlet
    pe = np.full(n_nodes, -1, dtype=np.int64)  # edge from the parent
    pe[v] = np.arange(E)
    parent = np.full(n_nodes, -1, dtype=np.int64)
    parent[v] = u
    depth = np.zeros(n_nodes, dtype=np.int64)
    order = [np.flatnonzero(parent < 0)]
    cs = np.argsort(u, kind="stable")
    cptr = np.concatenate([[0], np.cumsum(np.bincount(u, minlength=n_nodes))])
    while True:
        fr = order[-1]
        cnt = cptr[fr + 1] - cptr[fr]
        if cnt.sum() == 0:
            break
        idx = np.repeat(cptr[fr] - (np.cumsum(cnt) - cnt), cnt) + np.arange(cnt.sum())
        nxt = v[cs[idx]]
        depth[nxt] = len(order)
        order.append(nxt)
    phi_b = -np.asarray(p_bc(np.vstack([pos.T, np.zeros((3 - pos.shape[1], n_nodes))])), dtype=np.float64) * np.ones(n_nodes)
    leaf = deg == 1
    Ysum = np.zeros(n_nodes)  # sum of the children's equivalent conductances
    Yphi = np.zeros(n_nodes)  # sum of conductance * equivalent potential
    for lv_nodes in reversed(order[1:]):
        ge = g[pe[lv_nodes]]
        is_leaf = leaf[lv_nodes]
        ys = np.where(is_leaf, 1.0, Ysum[lv_nodes])
        Y = np.where(is_leaf, ge, ge * ys / (ge + ys))
        Phi = np.where(is_leaf, phi_b[lv_nodes], Yphi[lv_nodes] / ys)
        np.add.at(Ysum, parent[lv_nodes], Y)
        np.add.at(Yphi, parent[lv_nodes], Y * Phi)
    pot = np.zeros(n_nodes)
    root = order[0]
    pot[root] = phi_b[root]
    for lv_nodes in order[1:]:
        ge = g[pe[lv_nodes]]
        is_leaf = leaf[lv_nodes]
        pp = pot[parent[lv_nodes]]
        pot[lv_nodes] = np.where(is_leaf, phi_b[lv_nodes], (ge * pp + Yphi[lv_nodes]) / (ge + np.where(is_leaf, 1.0, Ysum[lv_nodes])))
    q_ref = g * (pot[u] - pot[v])
    lam_ref = pot[deg > 1]
    den_q, den_l = np.linalg.norm(q_ref), np.linalg.norm(lam_ref)
    return {"flux": float(np.linalg.norm(qg - q_ref) / den_q) if den_q > 0 else 0.0,
            "multipliers": float(np.linalg.norm(lg - lam_ref) / den_l) if den_l > 0 else 0.0}


def solution_blocks(solver):
    """Copies of the blocks of ``solver.x`` under the names of the Functions ``Solver.solve()`` returns."""
    asm = solver.assembler
    spaces = [*asm.flux_spaces, asm.pressure_space, asm.lm_space]
    names = [f"flux_color_{i}" for i in range(len(spaces) - 2)] + ["pressure", "global_flux"]
    solver.x.mark_device_modified()
    x = solver.x.array_r  # one D2H of the whole vector
    out, off = {}, 0
    for V, name in zip(spaces, names):
        out[name] = x[off:off + V.num_dofs].copy()
        off += V.num_dofs
    return out


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, max_bytes=DUMP_MAX_BYTES, seed=0):
    """``{name: array}`` -> ``out_dir/<name>.npy`` in float64, at most ``max_bytes`` in all (file headers
    included).  Beyond that every array keeps the same share of its entries, at sorted indices drawn by a
    generator seeded with ``seed``: arrays of the same sizes are always sampled at the same places."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(a, dtype=np.float64).ravel() for k, a in arrays.items()}
    data_bytes = sum(a.nbytes for a in arrays.values())
    budget = max_bytes - 128 * len(arrays)  # an .npy header is 128 bytes for a 1-D array
    share = min(1.0, budget / data_bytes) if data_bytes else 1.0
    for name, a in arrays.items():
        if share < 1.0:
            idx = np.random.default_rng(seed).choice(a.size, int(a.size * share), replace=False)
            a = a[np.sort(idx)]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def time_kernel(dev, fn, reps):
    fn()
    dev.sync()
    dev.timer_start()
    for _ in range(reps):
        fn()
    return dev.timer_stop() / reps


def load_traffic(n_dofs):
    """DRAM bytes per launch of the in-step kernels from THIS round's committed ``ncu --set full`` capture
    of the same workload (profiles/r2_traffic.json; ncu cannot run inside the bench)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            tj = json.load(fh)
        # (a rank of a partitioned weak-scaling run holds the same subtree plus a handful of replicated
        # multipliers: the per-GPU kernels move the same bytes to within that handful)
        if abs(tj["n_dofs_per_gpu"] - n_dofs) <= 64:
            return tj
    except (OSError, KeyError, ValueError):
        pass
    return None


def run_gpu(args):
    import ctypes as C

    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise RuntimeError("--dump-outputs writes the solution of a single-GPU run; run it without torchrun")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    N = args.cells_per_edge if args.cells_per_edge > 0 else 1
    n = args.generations
    if world > 1 and args.scaling == "weak":
        # weak scaling keeps ~one n-generation subtree per GPU: n + log2(world) generations
        n = args.generations + max(0, (world - 1).bit_length())
    pb = Problem(args.workload, n, N, local_rank, world, dist)
    nm, asm, solver, dev, ds = pb.nm, pb.asm, pb.solver, pb.dev, pb.ds
    n_dofs = asm.num_dofs
    n_dofs_total = pb.n_dofs_total
    if ds is not None:
        ds.assemble()
        ds.solve()
    else:
        solver.assemble()
        pb.functions = solver.create_functions()  # pinned result functions, reused by every e2e step
        solver.solve(pb.functions)
    nnz = solver.A.nnz
    E = nm.graph_edges.shape[0]
    nv = nm.mesh.topology.index_map(0).size_local
    n_bnd = nm.boundary_values.size

    sampler = ClockSampler(local_rank)
    sampler.start()  # sampled from warm-up to the end of the e2e loop (GPU under load throughout)
    ms_per_step, launches = pb.timed_steps(args.steps, args.warmup, barrier, dist, torch)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, solution_blocks(solver))
    value = n_dofs_total / (ms_per_step * 1e-3)
    opts, info, _lib = pb.opts, pb.info, pb._lib
    # true residual of the final iterate (one extra SpMV, outside the timed region)
    if ds is not None:
        hist = ds.solve(refine_steps=1, final_residual=True)
        rel_res, rel_res_final = hist[0], hist[-1]
        corrections = int(ds.corrections)
    else:
        rel_res = info.residual_norm / info.rhs_norm
        corrections = int(info.iterations) - 1
        opts_chk = solver.solve_options()
        opts_chk.final_residual = 1
        info_chk = _lib.SolveInfo()
        dev.call("nxfx_solve", solver.b.device_ptr(), solver.x.device_ptr_overwrite(), C.byref(opts_chk), C.byref(info_chk))
        rel_res_final = info_chk.residual_norm / info_chk.rhs_norm
    solver.x.mark_device_modified()
    t0 = time.perf_counter()
    parity = host_parity(pb, dist, torch)
    parity["host_seconds"] = time.perf_counter() - t0

    # ---- e2e through the Python API with host buffers --------------------------------------
    pbc_pinned = dev.pinned(nv)
    pbc_pinned[:] = asm._pbc_host
    x_host = dev.pinned(n_dofs) if ds is not None else None
    R_loc = ds._restrict(pb.R_edge, N, pb.G) if ds is not None else pb.R_edge
    f_loc = ds._restrict(pb.f_cell, N, pb.G) if ds is not None else pb.f_cell

    def step_e2e():
        asm.compute_forms(p_bc_ex=pbc_pinned, R=R_loc, f=f_loc)  # H2D of the boundary data (and coefficients)
        if ds is not None:
            ds.assemble()
            ds.solve()
            solver.x.d.download(x_host)  # D2H of the local part of the solution
            return
        solver.assemble()
        solver.solve(pb.functions)  # D2H of the solution blocks

    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    dev.sync()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = n_dofs_total * args.steps / e2e_s
    coef_bytes = sum(8 * np.size(c) for c in (R_loc, f_loc) if c is not None and not np.isscalar(c))
    # nvidia-smi needs ~0.2 s to deliver its first sample, the timed regions above are a few ms:
    # keep the GPU under the same load (untimed steps) until a handful of samples exist
    # (a fixed count derived from the all-reduced step time, so that all ranks stay in lock-step)
    for _ in range(min(5000, int(0.6 / max(ms_per_step * 1e-3, 1e-5)))):
        pb.step()
    dev.sync()
    clocks = sampler.stop()
    clocks["note"] = "sampled every 50 ms from warm-up until after the e2e loop, GPU kept under the timed load"

    # ---- per-kernel roofline (CUDA events on the launching stream) ---------------------------
    peak, peak_kind = measured_peaks()
    reps = 20
    solver.A.bind()
    xv, yv = solver.x, solver.b.duplicate()
    t_spmv = time_kernel(dev, lambda: dev.call("nxfx_spmv", xv.d.c_ptr, yv.d.c_ptr), reps)
    bytes_spmv = 12 * nnz + 4 * (n_dofs + 1) + 16 * n_dofs
    bdev = solver.b.duplicate()
    R_d, R_c = asm._R
    f_d, f_c = asm._f
    t_asm = time_kernel(
        dev, lambda: dev.call("nxfx_assemble", R_d.c_ptr if R_d is not None else None, C.c_double(R_c),
                              f_d.c_ptr if f_d is not None else None, C.c_double(f_c), 1, 1, 0, bdev.d.c_ptr), reps)
    bytes_asm = 24 * nv + 8 * nnz + 8 * n_dofs + 8 * n_bnd  # SURVEY 8(d): coords + values + rhs + p_bc
    kernel_ms = {"assemble": t_asm, "spmv": t_spmv}
    if ds is None:
        t_pcs = time_kernel(dev, lambda: dev.call("nxfx_pc_setup"), reps)
        t_pc = time_kernel(dev, lambda: dev.call("nxfx_pc_apply", solver.b.d.c_ptr, yv.d.c_ptr), reps)
        kernel_ms.update({"pc_apply": t_pc, "pc_setup": t_pcs})
    # the fused factor + first solve as run inside the step = step - assembly - residual (CUDA events)
    t_res = time_kernel(dev, lambda: dev.call("nxfx_residual", solver.b.d.c_ptr, xv.d.c_ptr, yv.d.c_ptr, None), reps) if ds is None else None
    gbs_spmv = bytes_spmv / (t_spmv * 1e-3) / 1e9
    gbs_asm = bytes_asm / (t_asm * 1e-3) / 1e9
    tj = load_traffic(n_dofs)
    tr = (lambda k: tj[k]["dram_bytes"] if tj and k in tj else None)
    n_bif = nm.bifurcation_values.size
    bytes_tree = 8 * n_dofs + 8 * E * N + 8 * n_bif  # reads r and R*h once, writes the multipliers
    t_tree = max(ms_per_step - t_asm - (t_res or t_spmv) - (tj["backsub"]["ms"] if tj and "backsub" in tj else 0.015), 1e-6)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": args.scaling if world > 1 else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": workload_name(args.workload, n, N), "n_dofs_total": n_dofs_total, "n_dofs_per_gpu": n_dofs, "nnz_per_gpu": nnz,
            "graph_edges_per_gpu": E,
            "solver": "preonly: network-Schur direct solve + 1 iterative-refinement step (residual of the first solve checked)",
            "relative_residual_before_refinement": rel_res, "relative_residual_final": rel_res_final,
            "refinement_corrections_per_step": corrections,
            "partition": (f"one {n}-generation tree cut into {world} edge partitions (subtrees); {ds.part.n_top} cut multipliers "
                          f"replicated; exchange = {pb.exchange}: "
                          + ("the top-chunk block of the fused tree kernel and the last block of the residual kernel store their "
                             "partial sums into every rank's buffer over NVLink (CUDA IPC), flag, wait, sum in rank order; no NCCL "
                             "call and one host sync per solve" if pb.exchange == "peer" else
                             "2 torch.distributed/NCCL all-reduces per solve between split kernel phases")) if world > 1 else "single GPU",
            "colouring": colouring_note(E, world),
            "l2": "per-step working set ~0.6 GB > 126 MB L2, no flush",
        },
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": (int(asm.pbc_h2d_bytes) + int(coef_bytes)) * world,
                "h2d_note": "p_bc: the caller hands over one value per mesh vertex; the forms read the boundary vertices only "
                            "(assembly.py:258-260), so only their contiguous id runs are copied",
                "d2h_bytes_per_step": int(8 * n_dofs) * world,
                "path": "assembler.compute_forms(p_bc array) + solver.assemble() + solver.solve(functions)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "parity": parity,
        "setup_ms": {**pb.setup_ms, "note": "host wall time per rank, once per network (the reference's Solve timer includes MUMPS "
                                            "analysis every solve; here the analysis is amortised over the steps)"},
        "roofline": {"kernel": "spmv_pipe_kernel<0> (CSR SpMV, TMA bulk pipeline)", "bound": "hbm", "achieved": gbs_spmv, "peak": peak,
                     "peak_kind": peak_kind, "unit": "GB/s", "frac": gbs_spmv / peak, "traffic": tr("residual"),
                     "traffic_kernel": "spmv_pipe_kernel<1> norms-only residual, the variant inside the step (profiles/r2_traffic.json)",
                     "algorithmic_bytes": bytes_spmv, "ms": t_spmv},
        "roofline_assembly": {"kernel": "assemble_tiles_kernel<false,true> (matrix + rhs, one launch)", "bound": "hbm", "achieved": gbs_asm, "peak": peak,
                              "peak_kind": peak_kind, "unit": "GB/s", "frac": gbs_asm / peak, "traffic": tr("assembly"),
                              "algorithmic_bytes": bytes_asm, "ms": t_asm},
        "roofline_tree": {"kernel": "tree_factor_solve_coop_kernel (factorisation fused with the first solve)", "bound": "hbm",
                          "achieved": bytes_tree / (t_tree * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": bytes_tree / (t_tree * 1e-3) / 1e9 / peak, "traffic": tr("tree"), "algorithmic_bytes": bytes_tree,
                          "ms": t_tree, "note": "ms = step - assembly - residual - back-substitution; the kernel is bound by the "
                                                "dependent level sweeps (latency), not by bandwidth"},
        "kernel_ms": kernel_ms,
    }
    # ---- strong scaling: the SAME fixed tree at every N (beside the weak-scaling headline) ----------
    if args.strong_generations > 0 and args.workload == "tree":
        del pb, solver, asm, nm, ds
        ns = args.strong_generations
        ps = Problem("tree", ns, 1, local_rank, world, dist)
        if ps.ds is not None:
            ps.ds.assemble()
            ps.ds.solve()
        else:
            ps.solver.assemble()
            ps.step()
        ms_s, launches_s = ps.timed_steps(max(5, args.steps // 2), 3, barrier, dist, torch)
        ps.solver.x.mark_device_modified()
        par_s = host_parity(ps, dist, torch)
        line["strong"] = {"workload": workload_name("tree", ns, 1), "n_dofs_total": ps.n_dofs_total, "ms_per_step": ms_s,
                          "value": ps.n_dofs_total / (ms_s * 1e-3), "unit": UNIT, "gpu_launches_per_step": launches_s / max(5, args.steps // 2),
                          "exchange": ps.exchange, "parity": {k: par_s[k] for k in ("true_residual_recomputed", "kirchhoff_max", "rel_l2_vs_closed_form")},
                          "note": "fixed problem size at every N: speed-up(N) = ms_per_step(1) / ms_per_step(N)"}
    # ---- higher-order elements (north_star item 1: P(k+1) flux / P(k) pressure): a side measurement ------------
    if world == 1 and args.higher_order_generations > 0 and args.workload == "tree":
        line["higher_order"] = higher_order_block(args.higher_order_generations, local_rank, max(3, args.steps // 4))
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.workload, n, N, steps=1, warmup=0)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def higher_order_block(n, device_index, steps):
    """P2/P1 and P3/P2 on make_tree(n), 4 cells per edge: table-driven assembly + the exact condensation (per-edge
    banded LU, 2 x 2 node blocks over the tree schedule) as ``preonly + lu`` -- one application and the residual
    check per step.  The residual is the solver's own true residual ||b - A x|| / ||b|| on the assembled CSR."""
    import ctypes as C

    import networks_fenicsx_b200 as nxfx
    from networks_fenicsx_b200 import _lib

    out = {"workload": f"make_tree(n={n},H={n},W={n}), N=4, smallest_last, direct solve (preonly + lu)"}
    for fd, pd in ((2, 1), (3, 2)):
        G = nxfx.network_generation.make_tree(n, float(n), float(n), as_arrays=True)
        nm = nxfx.NetworkMesh(G, N=4, color_strategy="smallest_last", device=device_index)
        asm = nxfx.HydraulicNetworkAssembler(nm, flux_degree=fd, pressure_degree=pd)
        asm.compute_forms(p_bc_ex=p_bc)
        solver = nxfx.Solver(asm)
        dev = nm.device
        opts, info = solver.solve_options(), _lib.SolveInfo()

        def step():
            solver.assemble()
            dev.call("nxfx_solve", solver.b.device_ptr(), solver.x.device_ptr_overwrite(), C.byref(opts), C.byref(info))

        step()
        l0 = dev.launch_count
        dev.timer_start()
        for _ in range(steps):
            step()
        ms = dev.timer_stop() / steps
        out[f"P{fd}/P{pd}"] = {"n_dofs": asm.num_dofs, "nnz": solver.A.nnz, "ms_per_step": ms, "value": asm.num_dofs / (ms * 1e-3),
                               "unit": UNIT, "relative_residual": info.residual_norm / info.rhs_norm,
                               "iterations": int(info.iterations), "gpu_launches_per_step": (dev.launch_count - l0) / steps}
        del solver, asm, nm
    return out


# ---- CPU baseline: the oracle port timed on the host ---------------------------------------------
def cpu_step_fn(workload, n, N=1):
    from networks_fenicsx_b200.mesh import _greedy_edge_coloring_arrays
    from oracle import reference_port as rp

    G, R, f = make_workload(workload, n, N)
    colors = _greedy_edge_coloring_arrays(G.number_of_nodes(), G.edges)
    net = rp.OracleNetwork(G.pos, G.edges, colors, N)
    pbc = net.eval_pbc(p_bc)
    Rc = 1.0 if R is None else np.repeat(R, N)
    fc = 0.0 if f is None else f

    def step():
        A, b = net.assemble(pbc, R=Rc, f=fc)
        return net.solve(A, b)

    return net, step


def cpu_baseline(workload, n, N, steps, warmup):
    net, step = cpu_step_fn(workload, n, N)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": net.n_dofs / dt, "unit": UNIT, "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
            "sample": f"{steps} step(s) of the full workload ({workload}, n={n}, {net.n_dofs} DOFs): NumPy COO->CSR assembly + "
                      f"SciPy SuperLU factor+solve (MUMPS stand-in; SuperLU is serial), {dt:.2f} s/step; 1 of {os.cpu_count()} host cores used"}


def run_reference(args):
    """--impl reference: the reference's own stack (DOLFINx/PETSc/MUMPS) cannot be installed here,
    so the oracle port is timed on the host cores, on the same config/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.generations
    N = args.cells_per_edge if args.cells_per_edge > 0 else 1
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and args.scaling == "weak":
        n += max(0, (world - 1).bit_length())  # same workload rule as the GPU arm
    # measured: 2.7 s per step at n = 20 (cost and memory grow linearly: x2 per generation); the
    # sample is bounded by ~150 s of CPU work and by n <= 21 (SuperLU memory at larger sizes)
    n_ref = min(n, 21)
    est = 3.0 * 2.0 ** (n_ref - 20) * N
    while n_ref > 10 and est * (args.steps + args.warmup) > 150.0:
        n_ref -= 1
        est /= 2.0
    net, step = cpu_step_fn(args.workload, n_ref, N)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = net.n_dofs / dt
    sample = (f"each step = full assemble+solve of {workload_name(args.workload, n_ref, N)} ({net.n_dofs} DOFs)"
              + ("" if n_ref == n else f" -- a bounded sample: the GPU arm's workload at this N is n={n}; DOFs/s is a rate, "
                                       f"CPU cost grows linearly with the tree size")
              + f": NumPy COO->CSR + SciPy SuperLU, 1 thread of {os.cpu_count()} host cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, n_ref, N), "workload_of_gpu_arm": workload_name(args.workload, n, N),
                   "same_config": n_ref == n},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "host_cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--generations", type=int, default=None)
    ap.add_argument("--workload", default="tree", choices=["tree", "arterial"])
    ap.add_argument("--cells-per-edge", type=int, default=0, help="default 1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = n + log2(N) generations (one ~20-generation subtree per GPU), strong = same tree")
    ap.add_argument("--higher-order-generations", type=int, default=16,
                    help="P2/P1 and P3/P2 side measurement on make_tree(m), N=4 (single GPU); 0 = skip")
    ap.add_argument("--strong-generations", type=int, default=23,
                    help="fixed tree of the extra strong-scaling block printed at every N (0 = off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the solution of the last timed step as DIR/<block>.npy (float64, single GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed; it needs --impl b200")
    if args.generations is None:
        args.generations = 20 if args.workload == "tree" else 18
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
