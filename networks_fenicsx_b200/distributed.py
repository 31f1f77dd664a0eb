"""Edge partition of ONE network over several GPUs (SURVEY 8e, north_star "each GPU owns an edge
partition; NCCL carries the bifurcation-node halo exchange and the all-reduces").

Partition = the elimination schedule's own structure (``schedule.py``): the bottom chunks
(complete subtrees) are dealt to the ranks in order, every graph edge follows its deeper
bifurcation, and the multipliers of the top chunk -- the cut bifurcations -- are REPLICATED on all
ranks.  Everything that couples ranks is additive and small (n_top doubles):

* ``y = A x``: the shared multiplier rows are partial sums -> one all-reduce;
* preconditioner: the top chunk's partial diagonal / right-hand side (contributions of each rank's
  chunk roots and incident edges) -> one all-reduce, then every rank eliminates the identical top
  chunk redundantly and back-substitutes its own chunks;
* norms: owned entries only, one all-reduce of the scalars.

Higher-order elements go the same way: the shared nodes carry 2 x 2 blocks {P_b, lam_b} (their
diagonal blocks, coupling blocks and nodal right-hand sides are exchanged), and with a continuous
pressure the nodal pressure rows of the shared bifurcations are partial sums like their multiplier
rows.  The section sizes come from the library (``nxfx_exchange_sizes``).

Host code (NumPy) in this file; collectives through one small seam: ``TorchDistGroup``
(``torch.distributed``: NCCL on GPUs, gloo in the CPU tests; one process per rank) or ``ThreadGroup``
(ranks that are threads of one process: ``PartitionedSolver``).
"""

from __future__ import annotations

import ctypes as C
import dataclasses
import functools
import gc
import queue
import threading
import weakref

import numpy as np

from .network_generation import ArrayGraph
from .schedule import CHUNK_NODES, TreeSchedule, assemble_schedule, assign_chunks, spanning_forest


@dataclasses.dataclass
class TreePartition:
    rank: int
    world: int
    graph: ArrayGraph  # local sub-network (nodes: endpoints of the local edges + all cut nodes)
    node_degree: np.ndarray  # GLOBAL degree of every local node
    global_nodes: np.ndarray  # local node -> global node
    global_edges: np.ndarray  # local edge -> global edge
    global_bif: np.ndarray  # local multiplier -> global multiplier index
    shared_lm: np.ndarray  # local multiplier indices of the replicated (shared) multipliers
    lam_weight: np.ndarray  # 1.0 where this rank counts the multiplier row in norms / -r_lambda
    schedule: TreeSchedule  # local elimination schedule; top chunk (this rank's private heavy nodes + the shared ones) last
    n_top: int  # number of SHARED multipliers (the exchanged part of the top chunk), identical on all ranks
    n_global_bif: int


def partition_tree(graph: ArrayGraph, world: int, rank: int, chunk_nodes: int = CHUNK_NODES) -> TreePartition:
    """Deterministic: every rank calls this with the same graph and gets its own part."""
    edges = np.asarray(graph.edges, dtype=np.int64)
    n_nodes = graph.number_of_nodes()
    u, v = edges[:, 0], edges[:, 1]
    deg_out = np.bincount(u, minlength=n_nodes)
    deg_in = np.bincount(v, minlength=n_nodes)
    degree = deg_in + deg_out
    bif = np.flatnonzero(degree > 1)
    n_bif = bif.size
    lm = np.full(n_nodes, -1, dtype=np.int64)
    lm[bif] = np.arange(n_bif)
    inlets = np.flatnonzero((degree == 1) & (deg_out == 1))
    parent, pedge, depth, chord = spanning_forest(edges, lm, n_bif, inlets)
    if chord.size:
        raise NotImplementedError("the multi-GPU partition needs a forest (no cycles among the bifurcations)")
    cn = chunk_nodes
    while True:
        chunk, n_chunks = assign_chunks(parent, depth, cn)
        if n_chunks - 1 >= world or cn <= 2:
            break
        cn //= 2
    n_bottom = n_chunks - 1
    if n_bottom < world:
        raise ValueError(f"network too small to cut into {world} parts")
    top = chunk == n_bottom
    rank_of_chunk = (np.arange(n_bottom) * world) // n_bottom
    # Heavy (top-chunk) nodes come in two kinds.  A heavy node all of whose bottom chunks went to ONE rank is
    # PRIVATE to that rank: it joins that rank's top chunk and nobody else sees it.  Only the heavy nodes
    # whose subtree spans several ranks are SHARED (replicated, exchanged): world - 1 nodes for a balanced
    # binary tree instead of the whole top of the elimination tree (7 instead of 2047 on 8 GPUs), so the
    # redundant top-chunk work and the exchanged payload stay constant as the number of GPUs grows.
    rmin = np.full(n_bif, world, dtype=np.int64)
    rmax = np.full(n_bif, -1, dtype=np.int64)
    rmin[~top] = rmax[~top] = rank_of_chunk[chunk[~top]]
    by_depth = np.argsort(depth, kind="stable")
    bounds = np.flatnonzero(np.diff(depth[by_depth])) + 1
    for lv in reversed(np.split(by_depth, bounds)):
        lv = lv[parent[lv] >= 0]
        np.minimum.at(rmin, parent[lv], rmin[lv])
        np.maximum.at(rmax, parent[lv], rmax[lv])
    shared_bif = top & (rmin != rmax)
    # shared nodes (and the edges between two of them) -> rank 0; private heavy nodes -> their rank
    owner_bif = np.where(shared_bif, 0, np.where(top, rmin, rank_of_chunk[np.minimum(chunk, n_bottom - 1)]))
    # every edge follows its deeper bifurcation
    a, b = lm[u], lm[v]
    da = np.where(a >= 0, depth[np.maximum(a, 0)], -1)
    db = np.where(b >= 0, depth[np.maximum(b, 0)], -1)
    deeper = np.where(db >= da, b, a)
    owner_edge = np.where(deeper >= 0, owner_bif[np.maximum(deeper, 0)], 0)
    ge = np.flatnonzero(owner_edge == rank)
    # local nodes: endpoints of the local edges and ALL shared nodes, ascending global id
    gn = np.unique(np.concatenate([edges[ge].ravel(), bif[shared_bif]]))
    local_of = np.full(n_nodes, -1, dtype=np.int64)
    local_of[gn] = np.arange(gn.size)
    attrs = {k: np.asarray(val)[ge] for k, val in graph.edge_attrs.items()}
    sub = ArrayGraph(np.asarray(graph.pos)[gn], local_of[edges[ge]], attrs)
    # local multipliers (ascending global node id, as NetworkMesh numbers them)
    lbif_nodes = gn[degree[gn] > 1]
    gb = lm[lbif_nodes]  # global multiplier index of every local multiplier
    lb_of_gb = np.full(n_bif, -1, dtype=np.int64)
    lb_of_gb[gb] = np.arange(gb.size)
    mine = shared_bif[gb] | (owner_bif[gb] == rank)
    if not np.all(mine):
        # a bifurcation of another rank's chunk can only appear here as the far end of one of our
        # edges, which the "deeper bifurcation" rule excludes on forests
        raise AssertionError("partition invariant violated")
    lpar = np.where(parent[gb] >= 0, lb_of_gb[np.maximum(parent[gb], 0)], -1)
    assert np.all((parent[gb] < 0) | (lpar >= 0)), "parent of a local multiplier is not local"
    ledge_of = np.full(edges.shape[0], -1, dtype=np.int64)
    ledge_of[ge] = np.arange(ge.size)
    lpedge = np.where(pedge[gb] >= 0, ledge_of[np.maximum(pedge[gb], 0)], -1)
    # my bottom chunks renumbered 0..k-1, the top chunk last
    my_chunks = np.flatnonzero(rank_of_chunk == rank)
    lchunk_of = np.full(n_chunks, -1, dtype=np.int64)
    lchunk_of[my_chunks] = np.arange(my_chunks.size)
    lchunk_of[n_bottom] = my_chunks.size
    lchunk = lchunk_of[chunk[gb]]
    assert np.all(lchunk >= 0)
    sched = assemble_schedule(lpar, lpedge, depth[gb], lchunk, my_chunks.size + 1, np.zeros(0, dtype=np.int32))
    shared = np.flatnonzero(shared_bif[gb])
    weight = np.where(shared_bif[gb] & (rank != 0), 0.0, 1.0)
    return TreePartition(rank, world, sub, degree[gn], gn, ge, gb, shared.astype(np.int32), weight, sched,
                         int(shared_bif.sum()), n_bif)


class TorchDistGroup:
    """The collectives of :class:`DistributedSolver` over ``torch.distributed`` (one process per rank)."""

    def __init__(self, group=None):
        import torch.distributed as dist

        self._dist, self.group = dist, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)

    def all_reduce(self, t) -> None:
        self._dist.all_reduce(t, group=self.group)

    def all_reduce_scalar(self, v: float, device) -> float:
        import torch

        t = torch.tensor([float(v)], dtype=torch.float64, device=device)
        self._dist.all_reduce(t, group=self.group)
        return float(t.item())

    def all_gather(self, out: list, t) -> None:
        self._dist.all_gather(out, t, group=self.group)

    def barrier(self) -> None:
        self._dist.barrier(group=self.group)


@dataclasses.dataclass
class _ThreadShared:
    barrier: threading.Barrier
    slots: list  # two rounds of per-rank slots, used alternately


class ThreadGroup:
    """The collectives of :class:`DistributedSolver` for ranks that are threads of ONE process (one
    ``ThreadGroup`` per rank, from :meth:`create`).

    * ``barrier``: a ``threading.Barrier`` with a timeout; :meth:`abort` (called when a rank raises) breaks it,
      so the other ranks raise ``threading.BrokenBarrierError`` instead of waiting.
    * ``all_reduce`` of a float64 CUDA tensor: every rank records an event on its stream, the ranks swap
      (pointer, event), each stream waits for all the events and ``nxfx_group_sum`` adds the inputs in rank
      order into a scratch buffer (bit-identical on every rank); a second swap of events keeps every input
      alive until all ranks have read it, then the sum is copied back.  The rank's torch current stream must
      be its library stream (``PartitionedSolver`` sets both).  A CPU tensor is summed on the host, in rank order.
    * scalars, ``all_gather`` and :meth:`gather_object`: plain Python.

    Every call is collective: all ranks make the same calls in the same order."""

    def __init__(self, shared: _ThreadShared, rank: int, world: int, timeout: float):
        self._sh, self.rank, self.world, self.timeout = shared, rank, world, timeout
        self._round = 0
        self._dev = None  # Device of this rank (bind), for nxfx_group_sum
        self._events = None
        self._scratch = None

    @classmethod
    def create(cls, world: int, timeout: float = 300.0) -> list["ThreadGroup"]:
        shared = _ThreadShared(threading.Barrier(world), [[None] * world, [None] * world])
        return [cls(shared, r, world, timeout) for r in range(world)]

    def bind(self, dev) -> None:
        self._dev = dev

    def barrier(self) -> None:
        self._sh.barrier.wait(self.timeout)

    def abort(self) -> None:
        self._sh.barrier.abort()

    def _swap(self, obj) -> list:
        """Every rank's ``obj``, in rank order.  Two alternating slot rounds: a rank can only come back to
        a round after every rank has passed the barrier of the round in between, i.e. has read this one."""
        slots = self._sh.slots[self._round & 1]
        self._round += 1
        slots[self.rank] = obj
        self.barrier()
        return list(slots)

    def gather_object(self, obj) -> list:
        return self._swap(obj)

    def all_reduce_scalar(self, v: float, device=None) -> float:
        total = 0.0
        for x in self._swap(float(v)):
            total += x
        return total

    def all_gather(self, out: list, t) -> None:
        for o, x in zip(out, self._swap(t.detach().cpu().clone())):
            o.copy_(x)

    def all_reduce(self, t) -> None:
        import torch

        if not t.is_cuda:
            parts = self._swap(t.detach().clone())
            total = parts[0].clone()
            for x in parts[1:]:
                total += x
            t.copy_(total)
            return
        assert t.dtype == torch.float64 and t.is_contiguous(), "all_reduce: contiguous float64 tensors only"
        n = t.numel()
        stream = torch.cuda.current_stream(t.device)
        if self._events is None:
            self._events = (torch.cuda.Event(), torch.cuda.Event())
        if self._scratch is None or self._scratch.numel() < n:
            self._scratch = torch.empty(max(n, 1), dtype=torch.float64, device=t.device)
        ready, done = self._events
        ready.record(stream)
        inputs = self._swap((t.data_ptr(), ready))
        for _, ev in inputs:
            stream.wait_event(ev)
        ptrs = (C.c_void_p * self.world)(*[p for p, _ in inputs])
        self._dev.call("nxfx_group_sum", ptrs, self.world, C.c_void_p(self._scratch.data_ptr()), n)
        done.record(stream)
        for ev in self._swap(done):
            stream.wait_event(ev)  # nobody overwrites an input another rank still reads
        t.copy_(self._scratch[:n])


def _collectives(group):
    return group if isinstance(group, ThreadGroup) else TorchDistGroup(group)


class DistributedSolver:
    """Assemble + solve of ONE network cut over the ranks of ``torch.distributed`` (one process per
    GPU), or over the threads of one process (``group`` a :class:`ThreadGroup`; see :class:`PartitionedSolver`).
    Mirrors ``Solver`` for the default options (network-Schur direct solve + iterative
    refinement); the collectives are three kinds of small SUM all-reduces (see module docstring).

    Args:
        graph: the GLOBAL network (every rank passes the same :class:`ArrayGraph`).
        N: cells per graph edge.
        p_bc_ex, f, R: as :meth:`HydraulicNetworkAssembler.compute_forms`; ``R``/``f`` arrays are given for
            the GLOBAL network (per graph edge or per cell) and restricted to the local edges here.
        exchange: ``"peer"``: the kernels exchange the partial sums themselves over NVLink (CUDA IPC peer
            memory, ``peer.cuh``) -- the single-GPU launch sequence, no NCCL call, one host sync per solve
            (needs every chunk of this rank co-resident in the cooperative tree kernel: up to ~21 generations
            per GPU); ``"nccl"``: split phases around ``torch.distributed`` all-reduces;
            ``"auto"``: peer when available.
        device: CUDA ordinal of this rank.
        group: a ``torch.distributed`` process group (None: the default one) or this rank's :class:`ThreadGroup`.
        flux_degree, pressure_degree: element degrees as in :class:`HydraulicNetworkAssembler` (the peer
            exchange is implemented for 1 / 0 only: other degrees use the all-reduces).
        stream: ``cudaStream_t`` (as an int) the library runs this rank on; None: the legacy default stream.
    """

    def __init__(self, graph: ArrayGraph, N: int, p_bc_ex, f=None, R=None, device: int = 0,
                 color_strategy="smallest_last", chunk_nodes: int = CHUNK_NODES, group=None,
                 exchange: str = "auto", flux_degree: int = 1, pressure_degree: int = 0, stream: int | None = None):
        from .assembly import HydraulicNetworkAssembler
        from .mesh import NetworkMesh, SerialComm
        from .solver import Solver

        comm = _collectives(group)
        self.part = part = partition_tree(graph, comm.world, comm.rank, chunk_nodes)
        # the sub-network is handed over explicitly (comm = serial): no second partitioning inside
        mesh = NetworkMesh(part.graph, N=N, color_strategy=color_strategy, device=device,
                           node_degree=part.node_degree, comm=SerialComm())
        if stream is not None:
            mesh.device.set_stream(stream)
        assembler = HydraulicNetworkAssembler(mesh, flux_degree=flux_degree, pressure_degree=pressure_degree)
        assembler.compute_forms(p_bc_ex=p_bc_ex, f=self._restrict(f, N, graph), R=self._restrict(R, N, graph))
        solver = Solver(assembler, schedule=part.schedule)
        self._attach(part, mesh, assembler, solver, comm, exchange)

    @classmethod
    def from_solver(cls, solver, part: TreePartition, group=None, exchange: str = "auto") -> "DistributedSolver":
        """Distributed layer for an existing ``Solver`` on one rank's part of a partitioned network
        (``NetworkMesh(G, N, comm=TorchDistComm())`` under torchrun: the reference-API path)."""
        self = cls.__new__(cls)
        self._attach(part, solver.assembler.network, solver.assembler, solver, _collectives(group), exchange)
        return self

    def _attach(self, part: TreePartition, mesh, assembler, solver, comm, exchange: str) -> None:
        import torch

        from . import _lib

        self._C, self._torch, self._comm = C, torch, comm
        self.rank, self.world = comm.rank, comm.world
        self.part = part
        self.mesh, self.assembler, self.solver = mesh, assembler, solver
        N = mesh.cells_per_edge
        device = mesh.device.index
        assert np.array_equal(part.global_nodes[self.mesh.bifurcation_values], part.global_nodes[
            np.flatnonzero(part.node_degree > 1)])
        self.dev = self.mesh.device
        if isinstance(comm, ThreadGroup):
            comm.bind(self.dev)
        shared = np.ascontiguousarray(part.shared_lm, dtype=np.int32)
        weight = np.ascontiguousarray(part.lam_weight, dtype=np.float64)
        self.dev.call("nxfx_set_shared", shared.size, _lib.as_i32p(shared), _lib.as_f64p(weight))
        cuda = torch.device("cuda", device)
        n_setup, n_apply, n_res = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        self.dev.call("nxfx_exchange_sizes", C.byref(n_setup), C.byref(n_apply), C.byref(n_res))
        self._n_apply = n_apply.value
        self._top = torch.zeros(n_setup.value + n_apply.value, dtype=torch.float64, device=cuda)  # [setup | apply]
        self._sh = torch.zeros(n_res.value, dtype=torch.float64, device=cuda)  # halo rows + 2 norm partials
        self._nrm = torch.zeros(2 * 40, dtype=torch.float64, device=cuda)
        self._r = self.dev.empty(self.assembler.num_dofs)
        self.n_dofs_global = int(self._allreduce_scalar(self._owned_dofs()))
        self.history: list[float] = []
        self.rhs_norm = float("nan")
        self.corrections = 0
        self.exchange = "nccl"
        if exchange not in ("auto", "peer", "nccl"):
            raise ValueError("exchange must be 'auto', 'peer' or 'nccl'")
        if exchange != "nccl":
            self._connect_peers(required=exchange == "peer")

    def _connect_peers(self, required: bool) -> None:
        """Peer exchange over NVLink (``peer.cuh``): every rank exports its exchange buffer as a CUDA IPC
        handle, the handles are all-gathered (the only use of the group on this path) and mapped; ranks
        that are threads of one process (``ThreadGroup``) swap their contexts instead and use each other's
        buffers directly.  All ranks agree on the outcome; any failure falls back to the host-driven
        all-reduces unless ``required``."""
        C, torch = self._C, self._torch
        handle = (C.c_ubyte * 64)()
        slot = C.c_int32(0)
        ok = 1
        try:
            self.dev.call("nxfx_comm_create", self.rank, self.world, C.cast(handle, C.c_void_p), C.byref(slot))
        except RuntimeError as exc:  # e.g. the schedule does not fit the cooperative kernel
            ok, err = 0, str(exc)
        cuda = self._top.device
        mine = torch.tensor(list(bytes(handle)) + [slot.value & 0xFF, (slot.value >> 8) & 0xFF, (slot.value >> 16) & 0xFF, ok],
                            dtype=torch.uint8, device=cuda)
        allh = [torch.empty_like(mine) for _ in range(self.world)]
        self._comm.all_gather(allh, mine)
        table = np.stack([t.cpu().numpy() for t in allh])
        if ok and table[:, 67].all() and (table[:, 64:67] == table[0, 64:67]).all():
            blob = np.ascontiguousarray(table[:, :64]).tobytes()
            try:
                if isinstance(self._comm, ThreadGroup):
                    ctxs = self._comm.gather_object(self.dev.handle.value)
                    self.dev.call("nxfx_comm_connect_local", (C.c_void_p * self.world)(*ctxs), self.world)
                else:
                    self.dev.call("nxfx_comm_connect", C.c_char_p(blob))
            except RuntimeError as exc:
                ok, err = 0, str(exc)
        else:  # keep this rank's own reason when it has one (e.g. a higher-order context)
            err = err if not ok else "a rank could not create its exchange buffer (or the slot sizes differ)"
            ok = 0
        if self._allreduce_scalar(float(ok)) == float(self.world):
            self.exchange = "peer"
            self._comm.barrier()  # every buffer is mapped and zeroed before the first flag is written
            return
        self.dev.call("nxfx_comm_destroy")
        if required:
            raise RuntimeError(f"peer exchange unavailable: {err if not ok else 'another rank failed'}")

    def _restrict(self, coef, N: int, graph: ArrayGraph):
        """Per-edge / per-cell coefficient arrays of the GLOBAL network -> this rank's edges (arrays that
        already have the local size, scalars and None pass through)."""
        if coef is None or np.isscalar(coef):
            return coef
        arr = np.asarray(coef, dtype=np.float64)
        E = graph.number_of_edges()
        ge = self.part.global_edges
        if arr.shape == (E,) and ge.size != E:
            return arr[ge]
        if arr.shape == (E * N,) and ge.size != E:
            return arr.reshape(E, N)[ge].ravel()
        return arr

    def _owned_dofs(self) -> int:
        # replicated: the multipliers of the shared nodes and, for a continuous pressure, their nodal pressures
        n_sh = self.part.n_top * (2 if self.assembler.degrees[1] >= 1 else 1)
        return int(self.assembler.num_dofs - n_sh + (n_sh if self.rank == 0 else 0))

    def _allreduce_scalar(self, v: float) -> float:
        return self._comm.all_reduce_scalar(v, self._top.device)

    def _ptr(self, t, offset: int = 0):
        return self._C.c_void_p(t.data_ptr() + 8 * offset)

    def assemble(self) -> None:
        self.solver.assemble()

    def _apply(self, r_ptr, z_ptr, add: int) -> None:
        top = self._ptr(self._top)
        self.dev.call("nxfx_pc_apply_begin", r_ptr, top)
        self._comm.all_reduce(self._top[: self._n_apply])
        self.dev.call("nxfx_pc_apply_end", r_ptr, z_ptr, top, add)

    def solve(self, refine_steps: int = 1, final_residual: bool = False, refine_rtol: float = 1e-13):
        """x = P^{-1} b, then iterative refinement while ``||b - A x|| > refine_rtol ||b||`` (at most
        ``refine_steps`` corrections; the all-reduced norms are identical on every rank, so all
        ranks take the same decision).  Returns the global relative residual norms that were
        evaluated.  Collectives: 1 (setup fused with the first application) + 1 per residual (halo rows
        and norm partials in one buffer) + 1 per correction."""
        dev = self.dev
        b = self.solver.b.device_ptr()
        x = self.solver.x.device_ptr_overwrite()
        if self.exchange == "peer":
            return self._solve_peer(b, x, refine_steps, final_residual, refine_rtol)
        # factorisation and first application share one all-reduce: the forward sweep of the bottom
        # chunks only needs their own factors
        top = self._ptr(self._top)  # [setup: partial pivots / blocks, link couplings | apply: partial rhs]
        dev.call("nxfx_pc_setup_apply_begin", b, top)
        self._comm.all_reduce(self._top)
        dev.call("nxfx_pc_setup_apply_end", b, x, top)
        self.history = []
        applied = 0
        while refine_steps > 0 or final_residual:
            self._residual(b, x, 0)
            vals = self._nrm[:2].cpu().numpy()  # synchronises; identical on all ranks
            self.rhs_norm = float(np.sqrt(vals[1]))
            rel = float(np.sqrt(vals[0]) / self.rhs_norm) if self.rhs_norm > 0 else 0.0
            self.history.append(rel)
            if applied >= refine_steps or (refine_rtol > 0 and rel <= refine_rtol) or not np.isfinite(rel):
                break
            self._apply(self._r.c_ptr, x, 1)
            applied += 1
            if applied >= refine_steps and not final_residual:
                break
        if not self.history:
            dev.sync()
        self.solver.x.mark_device_modified()
        self.corrections = applied
        return self.history

    def _solve_peer(self, b, x, refine_steps, final_residual, refine_rtol):
        """The single-GPU launch sequence (fused factor+solve tree kernel, back-substitution, residual)
        with the exchanges done inside the kernels over NVLink: one library call, one host
        synchronisation, no NCCL."""
        from . import _lib

        C = self._C
        key = (int(refine_steps), bool(final_residual), float(refine_rtol))
        cache = getattr(self, "_peer_opts", None)
        if cache is None or cache[0] != key:  # the option struct is built once: the step loop stays off the Python heap
            opts = self.solver.solve_options()
            opts.ksp_type, opts.pc_type = _lib.KSP_PREONLY, _lib.PC_NETWORK_SCHUR
            opts.refine_steps, opts.final_residual, opts.refine_rtol = key[0], int(key[1]), key[2]
            opts.error_if_not_converged = 0
            self._peer_opts = cache = (key, opts, _lib.SolveInfo())
        _, opts, info = cache
        self.solver.A._materialise_zero()
        self.solver.A.bind()
        self.dev.call("nxfx_solve", b, x, C.byref(opts), C.byref(info))
        self.solver.x.mark_device_modified()
        self.rhs_norm = float(info.rhs_norm)
        den = self.rhs_norm if self.rhs_norm > 0 else 1.0
        self.history = [info.history[i] / den for i in range(info.history_len)]
        self.corrections = int(info.iterations) - 1
        return self.history

    def _residual(self, b, x, k: int) -> None:
        """r = b - A x with consistent shared rows and the global [||r||^2, ||b||^2] in slot k:
        one all-reduce of the shared rows + 2 doubles."""
        dev = self.dev
        sh = self._ptr(self._sh)
        dev.call("nxfx_residual_partial", b, x, self._r.c_ptr, sh)
        self._comm.all_reduce(self._sh)
        dev.call("nxfx_residual_finish", sh, self._r.c_ptr, self._ptr(self._nrm, 2 * k))

    # ---- results -------------------------------------------------------------------------------
    def local_solution(self) -> np.ndarray:
        return self.solver.x.array_r

    def edge_values(self):
        """(global edge ids, flux[E_loc, N+1], pressure[E_loc, N]) of the local edges and
        (global multiplier ids, values) of the multipliers this rank owns."""
        x = self.local_solution()
        N = self.mesh.cells_per_edge
        E = self.part.global_edges.size
        fb = self.mesh.edge_slot.astype(np.int64) * (N + 1)
        q = x[fb[:, None] + np.arange(N + 1)[None, :]]
        nq = E * (N + 1)
        p = x[nq: nq + E * N].reshape(E, N)
        lam = x[nq + E * N:]
        own = self.part.lam_weight > 0
        return self.part.global_edges, q, p, self.part.global_bif[own], lam[own]

    def dof_values(self) -> dict:
        """The local solution in a form that places into the WHOLE network's numbering for any degree:

        * ``edges`` (global edge ids), ``flux`` ``[E_loc, fd N + 1]`` (the edge's vertex dofs, then the interior
          dofs cell by cell) and ``pressure`` ``[E_loc, k]``: DG0: the N cell values; continuous: the N - 1
          interior vertices, then the ``N (pd - 1)`` cell-interior dofs cell by cell;
        * ``nodes`` / ``node_pressure``: global node id and vertex pressure of the graph nodes this rank owns
          (continuous pressure; the nodal pressure of a shared bifurcation is owned by rank 0);
        * ``multipliers`` / ``lam``: global multiplier id and value of the multipliers this rank owns."""
        x = self.local_solution()
        N = self.mesh.cells_per_edge
        fd, pd = self.assembler.degrees
        ge = self.part.global_edges
        E = ge.size
        per_edge = fd * N + 1
        fb = self.mesh.edge_slot.astype(np.int64) * per_edge
        flux = x[fb[:, None] + np.arange(per_edge)[None, :]]
        nq = E * per_edge
        n_nodes = self.part.global_nodes.size
        e = np.arange(E)[:, None]
        if pd == 0:
            pressure = x[nq + e * N + np.arange(N)[None, :]]
            nodes = np.zeros(0, dtype=np.int64)
            node_p = np.zeros(0)
        else:
            nv = n_nodes + (N - 1) * E
            inner = nq + n_nodes + e * (N - 1) + np.arange(N - 1)[None, :]
            cell = nq + nv + e * (N * (pd - 1)) + np.arange(N * (pd - 1))[None, :]
            pressure = x[np.concatenate([inner, cell], axis=1)]
            shared_nodes = self.mesh.bifurcation_values[self.part.shared_lm]
            own = np.ones(n_nodes, dtype=bool)
            if self.rank != 0:
                own[shared_nodes] = False
            local = np.flatnonzero(own)
            nodes = self.part.global_nodes[local]
            node_p = x[nq + local]
        loff = x.size - self.part.global_bif.size
        own_lm = self.part.lam_weight > 0
        return {"edges": ge, "flux": flux, "pressure": pressure, "nodes": nodes, "node_pressure": node_p,
                "multipliers": self.part.global_bif[own_lm], "lam": x[loff:][own_lm]}


class _Worker:
    """One persistent thread of a :class:`PartitionedSolver`: the rank's device is current and its own
    non-blocking torch stream is the current stream for everything the thread runs."""

    def __init__(self, rank: int, device: int, on_error):
        self.rank, self.device, self._on_error = rank, device, on_error
        self.tasks: queue.SimpleQueue = queue.SimpleQueue()
        self.stream = None
        self.thread = threading.Thread(target=self._loop, name=f"nxfx-rank{rank}", daemon=True)
        self.thread.start()

    def _loop(self) -> None:
        setup_error = None
        try:
            import torch

            torch.cuda.set_device(self.device)
            # torch pool streams are created with cudaStreamNonBlocking: no implicit synchronisation with the legacy
            # stream of another thread (nxfx_comm_connect_local checks the flag)
            self.stream = torch.cuda.Stream(self.device)
            torch.cuda.set_stream(self.stream)
        except BaseException as exc:  # reported by every task
            setup_error = exc
        while True:
            item = self.tasks.get()
            if item is None:
                return
            fn, done = item
            if setup_error is not None:
                self._on_error()
                done.put((None, setup_error))
                continue
            try:
                done.put((fn(), None))
            except BaseException as exc:
                self._on_error()  # the other ranks leave their barriers instead of waiting for this one
                done.put((None, exc))


def _stop_workers(workers) -> None:
    for w in workers:
        w.tasks.put(None)
    for w in workers:
        w.thread.join()


class PartitionedSolver:
    """ONE network cut into ``len(devices)`` parts and solved from one process, without a launcher: one
    persistent worker thread per part, each with a :class:`DistributedSolver` on its own non-blocking stream
    of ``cuda:devices[rank]``, the ranks' collectives through a :class:`ThreadGroup`.  An entry of ``devices``
    may repeat (``devices=[0, 0]``: two parts on one GPU).

    ``exchange``: ``"peer"`` -- the kernels exchange the partial sums through each other's device memory (the
    single-GPU launch sequence; ranks on one device need their cooperative tree grids resident together);
    ``"nccl"`` -- the split phases around the group's all-reduce (``nxfx_group_sum``); ``"auto"`` -- peer when
    available.  :attr:`exchange` reports the mode the ranks agreed on.

    ``assemble()`` / ``solve()`` run on every rank at once; ``solve`` returns rank 0's residual history (identical
    on every rank).  An exception in any rank stops every thread and is re-raised here.  Use as a context
    manager or call :meth:`close`."""

    def __init__(self, graph: ArrayGraph, N: int, p_bc_ex, f=None, R=None, devices=(0, 1), flux_degree: int = 1,
                 pressure_degree: int = 0, exchange: str = "auto", chunk_nodes: int = CHUNK_NODES,
                 timeout: float = 300.0):
        devices = [int(d) for d in devices]
        if not devices:
            raise ValueError("devices must name at least one GPU")
        groups = ThreadGroup.create(len(devices), timeout)
        self._workers = [_Worker(r, d, groups[0].abort) for r, d in enumerate(devices)]
        self._finalizer = weakref.finalize(self, _stop_workers, self._workers)
        self.devices = devices
        self.solvers: list[DistributedSolver | None] = [None] * len(devices)

        def build(rank):
            w = self._workers[rank]
            self.solvers[rank] = DistributedSolver(
                graph, N, p_bc_ex, f=f, R=R, device=w.device, chunk_nodes=chunk_nodes, group=groups[rank],
                exchange=exchange, flux_degree=flux_degree, pressure_degree=pressure_degree,
                stream=w.stream.cuda_stream)

        self._run(build)

    def _run(self, fn) -> list:
        """fn(rank) on every rank's thread at once; the results in rank order."""
        if not self._finalizer.alive:
            raise RuntimeError("PartitionedSolver is closed")
        done = [queue.SimpleQueue() for _ in self._workers]
        for w, d in zip(self._workers, done):
            w.tasks.put((functools.partial(fn, w.rank), d))
        results = [d.get() for d in done]
        errors = [e for _, e in results if e is not None]
        if errors:
            self.close()
            # the first failure, not the broken barriers it caused in the other ranks
            raise next((e for e in errors if not isinstance(e, threading.BrokenBarrierError)), errors[0])
        return [r for r, _ in results]

    def map(self, fn) -> list:
        """fn(DistributedSolver) on every rank's thread (its device and stream current); the results in rank order."""
        return self._run(lambda rank: fn(self.solvers[rank]))

    @property
    def exchange(self) -> str:
        return self.solvers[0].exchange

    def assemble(self) -> None:
        self.map(lambda s: s.assemble())

    def solve(self, refine_steps: int = 1, final_residual: bool = False, refine_rtol: float = 1e-13) -> list[float]:
        return self.map(lambda s: s.solve(refine_steps, final_residual, refine_rtol))[0]

    def dof_values(self) -> list[dict]:
        """Every rank's :meth:`DistributedSolver.dof_values` (global edge, node and multiplier ids)."""
        return self.map(lambda s: s.dof_values())

    def close(self) -> None:
        """Release every rank's solver on its own thread, then stop and join the threads."""
        if not self._finalizer.alive:
            return
        done = [queue.SimpleQueue() for _ in self._workers]
        for w, d in zip(self._workers, done):
            w.tasks.put((functools.partial(self._release, w.rank), d))
        for d in done:
            d.get()
        self._finalizer()

    def _release(self, rank: int) -> None:
        self.solvers[rank] = None
        gc.collect()

    def __enter__(self) -> "PartitionedSolver":
        return self

    def __exit__(self, *exc) -> None:
        self.close()
