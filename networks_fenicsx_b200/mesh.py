"""Graph -> network mesh (drop-in for ``networks_fenicsx.mesh.NetworkMesh``, mesh.py:45-538).

Host side (this file, NumPy, vectorised): graph analysis (mesh.py:175-225), colouring
(mesh.py:29-42), dof-slot layout, bifurcation incidence tables.  Device side (libnxfx_b200):
vertex coordinates (mesh.py:270-292), everything downstream.  DOLFINx objects are replaced by
small duck types that answer the attributes the reference's tests, demos and post-processing
touch (SURVEY section 4): ``mesh.topology.dim``, ``mesh.geometry.dim/x``,
``topology.index_map(d).size_global``, ``subdomains``/``boundaries`` mesh tags, ``submeshes``,
``entity_maps``, ``orientation``, ``in_edges``/``out_edges``, ``lm_mesh``.

Numbering is the canonical serial numbering (DESIGN.md): cell ``e*N + j`` for the j-th cell of
graph edge e (``graph.edges()`` order, running u -> v), vertices = graph nodes followed by the
``N-1`` interior points of every edge.
"""

from __future__ import annotations

import ctypes as C
from typing import Callable, Iterable

import numpy as np
import numpy.typing as npt

from . import _lib
from .common import timed
from .device import Device, DeviceArray
from .network_generation import ArrayGraph

__all__ = ["NetworkMesh", "color_graph"]

# Colouring regimes (mesh.py:38-39 calls networkx on the line graph: minutes and gigabytes at a million edges):
#   <= NETWORKX_COLORING_MAX_EDGES          networkx itself (any strategy, callables included)
#   <= NETWORKX_IDENTICAL_MAX_EDGES         'smallest_last' / 'largest_first' reproduced edge by edge
#                                           (_networkx_identical_edge_coloring), ~26 s at a million edges
#   beyond, or other strategies at scale    native greedy colouring in input order + a warning: the flux
#                                           block layout is then a permutation of the reference's
NETWORKX_COLORING_MAX_EDGES = 70_000
NETWORKX_IDENTICAL_MAX_EDGES = 2_200_000


class SerialComm:
    """Stand-in for ``MPI.COMM_WORLD`` on one process (mesh.py:89)."""

    rank = 0
    size = 1

    def allreduce(self, value, op=None):
        return value

    def bcast(self, value, root=0):
        return value

    def barrier(self):
        return None

    Get_rank = lambda self: 0  # noqa: E731
    Get_size = lambda self: 1  # noqa: E731


COMM_WORLD = SerialComm()


def _resolve_comm(comm):
    """The reference defaults to ``MPI.COMM_WORLD`` (mesh.py:89), so the same script runs serially or
    under ``mpiexec -n k``.  Here the launcher is ``torchrun``: with ``comm=None`` and ``WORLD_SIZE > 1`` in
    the environment the process group is initialised (NCCL, one GPU per local rank) and a
    ``TorchDistComm`` is returned; otherwise the serial stand-in."""
    import os

    if comm is not None:
        return comm
    if int(os.environ.get("WORLD_SIZE", "1")) <= 1:
        return COMM_WORLD
    import torch
    import torch.distributed as dist

    from .parallel import TorchDistComm

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if torch.cuda.is_available():
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        else:
            dist.init_process_group("gloo")
    return TorchDistComm(device=torch.device("cuda", local_rank) if torch.cuda.is_available() else None)


# --------------------------------------------------------------------------------------------
# colouring (mesh.py:29-42)
# --------------------------------------------------------------------------------------------
def _greedy_edge_coloring_arrays(n_nodes: int, edges: np.ndarray) -> np.ndarray:
    """Proper greedy edge colouring without networkx: edges are visited in input order and take
    the smallest colour not used at either endpoint.  max-degree colours on forests whose edges
    are listed parent-first (all generators here), at most 2*maxdeg-1 in general."""
    E = edges.shape[0]
    deg = np.bincount(edges.ravel(), minlength=n_nodes)
    maxc = int(2 * deg.max())
    colors = np.full(E, -1, dtype=np.int32)
    if maxc <= 62:
        used = np.zeros(n_nodes, dtype=np.int64)  # bitmask of colours used at each node
        u_all, v_all = edges[:, 0], edges[:, 1]
        # process in rounds of mutually non-adjacent edges: an edge is ready when it is the
        # lowest-index uncoloured edge at both of its endpoints
        remaining = np.arange(E)
        rounds = 0
        while remaining.size:
            rounds += 1
            if rounds > 64 and remaining.size > 1024:
                # long chains (path-like graphs): a round colours a handful of edges only -- O(E) rounds of O(E)
                # work.  Finish sequentially; same visiting order, same result.
                used_l = used.tolist()
                for e, u, v in zip(remaining.tolist(), u_all[remaining].tolist(), v_all[remaining].tolist()):
                    free = ~(used_l[u] | used_l[v])
                    low = free & -free
                    colors[e] = low.bit_length() - 1
                    used_l[u] |= low
                    used_l[v] |= low
                return colors
            first_at = np.full(n_nodes, E, dtype=np.int64)
            np.minimum.at(first_at, u_all[remaining], remaining)
            np.minimum.at(first_at, v_all[remaining], remaining)
            ready = remaining[(first_at[u_all[remaining]] == remaining) & (first_at[v_all[remaining]] == remaining)]
            mask = used[u_all[ready]] | used[v_all[ready]]
            free = ~mask
            lowest = free & -free  # lowest zero bit of mask
            col = np.round(np.log2(lowest.astype(np.float64))).astype(np.int32)
            colors[ready] = col
            used[u_all[ready]] |= lowest
            used[v_all[ready]] |= lowest
            remaining = remaining[colors[remaining] < 0]
        return colors
    used_sets = [set() for _ in range(n_nodes)]
    for e, (u, v) in enumerate(edges.tolist()):
        c = 0
        while c in used_sets[u] or c in used_sets[v]:
            c += 1
        colors[e] = c
        used_sets[u].add(c)
        used_sets[v].add(c)
    return colors


def _as_strategy_name(strategy) -> str | None:
    """'smallest_last' / 'largest_first' for the strings and for networkx's own strategy functions."""
    if isinstance(strategy, str):
        return strategy
    name = getattr(strategy, "__name__", "")
    if getattr(strategy, "__module__", "").startswith("networkx.") and name.startswith("strategy_"):
        return name[len("strategy_"):]
    return None


def _networkx_identical_edge_coloring(n_nodes: int, edges: np.ndarray, strategy: str) -> np.ndarray:
    """The colouring ``nx.coloring.greedy_color(nx.line_graph(G.to_undirected()), strategy)`` assigns
    (mesh.py:38-39), edge by edge IDENTICAL to networkx 3.x, without building networkx graphs.

    What networkx returns depends on iteration orders: ``line_graph`` collects the line-graph edges in a
    Python ``set`` of tuple pairs and adds them in the set's iteration order (which fixes the node and
    adjacency order of the line graph), and ``smallest_last`` pops nodes from per-degree ``set`` buckets.
    Both are reproduced by running the SAME sequence of operations on real CPython sets holding the same
    tuples (the iteration order of a set is a function of its elements' hashes and its insertion
    history), while everything else is flat lists -- about 4x faster and 3x smaller than networkx at a
    million edges.  ``largest_first`` is a stable sort by line-graph degree.  Checked against networkx
    on trees, arterial trees and random graphs in tests/test_host_logic.py."""
    import itertools
    from collections import defaultdict, deque

    E = edges.shape[0]
    # G.to_undirected() walks the directed edges grouped by source node (node order), successors in
    # insertion order; nodes are 0..n-1 in order, so their index is their value
    order = np.argsort(edges[:, 0], kind="stable")
    el = edges[order].tolist()
    adj: list[list[int]] = [[] for _ in range(n_nodes)]
    seen_pair = set()
    for u, v in el:
        key = (u, v) if u < v else (v, u)
        if key in seen_pair:
            raise ValueError("antiparallel / duplicate edges: use networkx for this graph")
        seen_pair.add(key)
        adj[u].append(v)
        adj[v].append(u)
    del seen_pair
    # nx.generators.line._lg_undirected
    lnodes: dict[tuple[int, int], int] = {}  # line-graph node -> index in L's node order
    pairs: set = set()
    for u in range(n_nodes):
        nodes = [(u, w) if u < w else (w, u) for w in adj[u]]
        if len(nodes) == 1 and nodes[0] not in lnodes:
            lnodes[nodes[0]] = len(lnodes)
        for i, a in enumerate(nodes):
            pairs.update([(a, b) if a < b else (b, a) for b in nodes[i + 1:]])
    ladj: list[list[int]] = [[] for _ in range(E)]
    for a, b in pairs:  # L.add_edges_from(edges): set iteration order
        ia = lnodes.get(a)
        if ia is None:
            ia = lnodes[a] = len(lnodes)
        ib = lnodes.get(b)
        if ib is None:
            ib = lnodes[b] = len(lnodes)
        ladj[ia].append(ib)
        ladj[ib].append(ia)
    del pairs
    if len(lnodes) != E:
        raise AssertionError("line graph has a different number of nodes than the graph has edges")
    keys = list(lnodes)  # node tuples in L's node order
    deg = [len(x) for x in ladj]
    if strategy == "largest_first":  # sorted(G, key=G.degree, reverse=True): stable
        seq = np.argsort(-np.asarray(deg, dtype=np.int64), kind="stable").tolist()
    elif strategy == "smallest_last":
        degrees: dict = defaultdict(set)
        lbound = float("inf")
        for i, d in enumerate(deg):
            degrees[d].add(keys[i])
            lbound = min(lbound, d)
        # the strategy works on H = G.copy(): the copy re-adds the edges walking the nodes in order, so in
        # H a node's neighbours that precede it in node order come first (ascending), then the others in
        # their original adjacency order
        hadj = [sorted(w for w in nb if w < i) + [w for w in nb if w > i] for i, nb in enumerate(ladj)]
        alive = [True] * E
        result: deque = deque()
        for _ in range(E):
            min_degree = next(d for d in itertools.count(lbound) if d in degrees)
            bucket = degrees[min_degree]
            u = lnodes[bucket.pop()]
            if not bucket:
                del degrees[min_degree]
            result.appendleft(u)
            for v in hadj[u]:
                if not alive[v]:
                    continue
                d = deg[v]
                b = degrees[d]
                b.remove(keys[v])
                if not b:
                    del degrees[d]
                degrees[d - 1].add(keys[v])
                deg[v] = d - 1
            alive[u] = False
            lbound = min_degree - 1
        seq = list(result)
    else:
        raise ValueError(f"strategy {strategy!r} is not reproduced natively")
    # nx.coloring.greedy_color: first colour not used by an already coloured neighbour
    col = [-1] * E
    for u in seq:
        used = {col[v] for v in ladj[u] if col[v] >= 0}
        c = 0
        while c in used:
            c += 1
        col[u] = c
    out = np.empty(E, dtype=np.int32)
    ekey = [(u, v) if u < v else (v, u) for u, v in edges.tolist()]
    out[:] = [col[lnodes[k]] for k in ekey]
    return out


@timed("nxfx:color_graph")
def color_graph(
    graph,
    strategy: str | Callable | None,
) -> dict[tuple[int, int], int]:
    """Colour the edges of a graph (mesh.py:29-42).

    ``strategy=None``: colour = index of the edge in ``graph.edges`` (one flux space per edge).
    Otherwise the reference's call sequence -- greedy colouring of the line graph of the undirected
    graph with networkx -- is used verbatim up to ``NETWORKX_COLORING_MAX_EDGES`` edges; up to
    ``NETWORKX_IDENTICAL_MAX_EDGES`` the strategies ``smallest_last`` / ``largest_first`` are reproduced
    edge by edge without networkx graphs; beyond that a native greedy colouring is used and a warning
    says so (same number of colours on trees, not the same assignment).
    """
    edges = _edge_array(graph)
    if strategy is None:
        return {(int(u), int(v)): i for i, (u, v) in enumerate(edges.tolist())}
    if edges.shape[0] <= NETWORKX_COLORING_MAX_EDGES:
        import networkx as nx

        G = graph.to_networkx() if isinstance(graph, ArrayGraph) else graph
        return nx.coloring.greedy_color(nx.line_graph(G.to_undirected()), strategy=strategy)
    col = _large_graph_colors(graph.number_of_nodes(), edges, strategy)
    return {(int(u), int(v)): int(c) for (u, v), c in zip(edges.tolist(), col.tolist())}


def _large_graph_colors(n_nodes: int, edges: np.ndarray, strategy) -> np.ndarray:
    """Colours of a graph too large for networkx itself: networkx-identical where that is reproduced,
    else the native greedy colouring -- never silently: the caller is told when the strategy it asked
    for is not the one it gets."""
    import warnings

    name = _as_strategy_name(strategy)
    E = edges.shape[0]
    if name in ("smallest_last", "largest_first") and E <= NETWORKX_IDENTICAL_MAX_EDGES:
        try:
            return _networkx_identical_edge_coloring(n_nodes, edges, name)
        except ValueError as exc:  # antiparallel edges
            warnings.warn(f"networkx-identical colouring not available ({exc}); using the native greedy colouring",
                          stacklevel=3)
    else:
        warnings.warn(
            f"color_strategy={name or strategy!r} on {E} graph edges: beyond "
            f"{NETWORKX_IDENTICAL_MAX_EDGES if name in ('smallest_last', 'largest_first') else NETWORKX_COLORING_MAX_EDGES} "
            "edges the requested networkx strategy is replaced by a native greedy colouring in input order "
            "(same number of colours on trees; the flux blocks are a permutation of the reference's layout)",
            stacklevel=3)
    return _greedy_edge_coloring_arrays(n_nodes, edges)


def _edge_array(graph) -> np.ndarray:
    if isinstance(graph, ArrayGraph):
        return np.asarray(graph.edges, dtype=np.int64).reshape(-1, 2)
    return np.asarray(list(graph.edges()), dtype=np.int64).reshape(-1, 2)


def _edge_colors(graph, strategy, edges: np.ndarray) -> np.ndarray:
    """Colour per edge in ``graph.edges()`` order (array form of ``color_graph``); the lookup is
    insensitive to the (u, v) / (v, u) keying of networkx line graphs (SURVEY Appendix D)."""
    E = edges.shape[0]
    if strategy is None:
        return np.arange(E, dtype=np.int32)
    if isinstance(strategy, np.ndarray):  # precomputed colours, one per edge in graph.edges() order (extension)
        col = np.ascontiguousarray(strategy, dtype=np.int32)
        if col.shape != (E,):
            raise ValueError("a colour array must have one entry per graph edge")
        return col
    if E > NETWORKX_COLORING_MAX_EDGES:
        return _large_graph_colors(graph.number_of_nodes(), edges, strategy)
    coloring = color_graph(graph, strategy)
    out = np.empty(E, dtype=np.int32)
    for i, (u, v) in enumerate(edges.tolist()):
        c = coloring.get((u, v))
        out[i] = coloring[(v, u)] if c is None else c
    return out


# --------------------------------------------------------------------------------------------
# duck types for the DOLFINx objects the reference exposes
# --------------------------------------------------------------------------------------------
class AdjacencyList:
    """``dolfinx.graph.AdjacencyList`` stand-in (mesh.py:258-263)."""

    def __init__(self, array, offsets):
        self.array = np.asarray(array, dtype=np.int32)
        self.offsets = np.asarray(offsets, dtype=np.int32)

    def links(self, i) -> npt.NDArray[np.int32]:
        i = int(i)
        return self.array[self.offsets[i] : self.offsets[i + 1]]

    @property
    def num_nodes(self) -> int:
        return self.offsets.size - 1


class IndexMap:
    def __init__(self, n: int):
        self.size_local = int(n)
        self.size_global = int(n)
        self.num_ghosts = 0
        self.local_range = (0, int(n))


class Topology:
    def __init__(self, dim: int, counts: dict[int, int], cells_fn=None):
        self.dim = dim
        self._counts = counts
        self._cells_fn = cells_fn

    def index_map(self, d: int) -> IndexMap:
        return IndexMap(self._counts[d])

    def create_connectivity(self, d0: int, d1: int) -> None:
        return None

    def create_entity_permutations(self) -> None:
        return None

    def connectivity(self, d0: int, d1: int):
        if d0 == self.dim and d1 == 0 and self._cells_fn is not None:
            cells = self._cells_fn()
            return AdjacencyList(cells.ravel(), np.arange(0, cells.size + 1, cells.shape[1]))
        raise NotImplementedError(f"connectivity({d0}, {d1})")


class Geometry:
    def __init__(self, dim: int, x_fn):
        self.dim = dim
        self._x_fn = x_fn

    @property
    def x(self) -> npt.NDArray[np.float64]:
        """Vertex coordinates, shape (n_vertices, 3), zero padded (DOLFINx convention)."""
        return self._x_fn()


class Mesh:
    """Minimal ``dolfinx.mesh.Mesh`` stand-in."""

    def __init__(self, comm, topology: Topology, geometry: Geometry, name="mesh"):
        self.comm = comm
        self.topology = topology
        self.geometry = geometry
        self.name = name

    def ufl_domain(self):
        return self


class MeshTags:
    """``dolfinx.mesh.MeshTags`` stand-in (indices sorted ascending)."""

    def __init__(self, mesh: Mesh, dim: int, indices, values, name=""):
        self.mesh = mesh
        self.dim = dim
        self.indices = np.asarray(indices, dtype=np.int32)
        self.values = np.asarray(values)
        self.name = name

    def find(self, value) -> npt.NDArray[np.int32]:
        return self.indices[self.values == value]


class EntityMap:
    """``dolfinx.mesh.EntityMap`` stand-in: sub entity i <-> parent entity ``sub_to_parent[i]``."""

    def __init__(self, sub_to_parent, n_parent: int):
        self._s2p = np.asarray(sub_to_parent, dtype=np.int32)
        self._n_parent = int(n_parent)
        self._p2s = None

    def sub_topology_to_topology(self, entities, inverse: bool = False):
        entities = np.asarray(entities, dtype=np.int32)
        if not inverse:
            return self._s2p[entities]
        if self._p2s is None:
            self._p2s = np.full(self._n_parent, -1, dtype=np.int32)
            self._p2s[self._s2p] = np.arange(self._s2p.size, dtype=np.int32)
        return self._p2s[entities]


class _LazyList:
    """List-like whose items are built on first access (one submesh per colour: with
    ``color_strategy=None`` there are as many colours as graph edges, mesh.py:438)."""

    def __init__(self, n: int, build: Callable[[int], object]):
        self._n = n
        self._build = build
        self._cache: dict[int, object] = {}

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        if i not in self._cache:
            self._cache[i] = self._build(i)
        return self._cache[i]

    def __iter__(self):
        return (self[i] for i in range(self._n))


class OrientationFunction:
    """DG0 orientation field (mesh.py:365-400).  The input sign (+1 iff the cell's first node index
    is smaller, mesh.py:321-322) is flipped back wherever the created cell is not ascending in
    input index (mesh.py:379-398); cells keep their u -> v node order, so the net value is +1 on
    every cell and ``orientation * t`` is the unit tangent of the graph edge."""

    name = "orientation"

    def __init__(self, n_cells: int, cells_fn):
        self._n = n_cells
        self._cells_fn = cells_fn
        self._arr = None
        self.x = self

    @property
    def array(self) -> npt.NDArray[np.float64]:
        if self._arr is None:
            cells = self._cells_fn()
            ascending = cells[:, 0] < cells[:, 1]
            s_in = np.where(ascending, 1.0, -1.0)
            self._arr = np.where(ascending, s_in, -s_in)
        return self._arr

    def scatter_forward(self):
        return None


# --------------------------------------------------------------------------------------------
class NetworkMesh:
    """Drop-in for ``networks_fenicsx.NetworkMesh`` (mesh.py:45-96).

    Args:
        graph: ``networkx.DiGraph`` whose nodes ``0..n-1`` carry ``"pos"`` (as the reference
            requires, mesh.py:177,183-184,274), or an :class:`ArrayGraph`.
        N: number of cells per graph edge.
        color_strategy: ``None`` (one flux space per edge) or a networkx greedy-colouring strategy.
        comm: kept for signature compatibility (single process per GPU).
        graph_rank: kept for signature compatibility.
        device: CUDA device ordinal (extension; default 0).
        node_degree: degree of every node in the GLOBAL graph when ``graph`` is one rank's part of
            a partitioned network (extension, see ``distributed.py``): a cut bifurcation keeps its
            multiplier although it may have a single local edge.
    """

    def __init__(
        self,
        graph,
        N: int,
        color_strategy: str | Callable | Iterable | None = None,
        comm=None,
        graph_rank: int = 0,
        device: int | Device | None = None,
        node_degree: npt.NDArray[np.integer] | None = None,
    ):
        self._node_degree_override = node_degree
        self._comm = comm = _resolve_comm(comm)
        self._device_arg = device
        self._partition = None  # this rank's part when the network is cut over several processes
        self._global_graph = None
        if getattr(comm, "size", 1) > 1 and node_degree is None:
            graph, node_degree = self._partition_over(comm, graph, N)
            self._node_degree_override = node_degree
            if device is None:
                import os

                self._device_arg = int(os.environ.get("LOCAL_RANK", "0"))
        self._dev: Device | None = None
        self._x_host = None
        self._cells_host = None
        self._build_mesh(graph, N=N, color_strategy=color_strategy, comm=comm, graph_rank=graph_rank)
        self._build_network_submeshes()
        self._create_lm_submesh()

    def _partition_over(self, comm, graph, N):
        """Several processes (torchrun; the reference: ``mpiexec``, mesh.py:227-250 distributes the mesh):
        every rank holds the whole graph (the reference builds it on ``graph_rank`` and lets DOLFINx
        distribute the cells) and keeps its edge partition of it -- subtrees of the elimination schedule,
        cut multipliers replicated (``distributed.partition_tree``).  Networks too small to cut, or with
        cycles, are REPLICATED: every rank then solves the whole network redundantly, with identical
        results.  Returns the graph this rank meshes and the global degrees of its nodes."""
        import warnings

        from .distributed import partition_tree

        if isinstance(graph, ArrayGraph):
            glob = graph
        else:
            nodes = np.fromiter(graph.nodes(), dtype=np.int64, count=graph.number_of_nodes())
            if not np.array_equal(nodes, np.arange(nodes.size)):
                raise ValueError("graph nodes must be the integers 0..n-1 in insertion order (mesh.py:183-184,274)")
            attrs = {}
            edges = _edge_array(graph)
            if edges.shape[0] and all("radius" in graph.edges[e] for e in graph.edges()):
                attrs["radius"] = np.asarray([graph.edges[e]["radius"] for e in graph.edges()], dtype=np.float64)
            glob = ArrayGraph(np.asarray([graph.nodes[v]["pos"] for v in graph.nodes()], dtype=np.float64), edges, attrs)
        self._global_graph = glob
        try:
            part = partition_tree(glob, comm.size, comm.rank)
        except (ValueError, NotImplementedError) as exc:
            if comm.rank == 0:
                warnings.warn(f"the network is not cut over the {comm.size} processes ({exc}): every rank solves all of it",
                              stacklevel=3)
            return graph, None
        self._partition = part
        return part.graph, part.node_degree

    # ---- host-side graph analysis ---------------------------------------------------------
    @timed("nxfx:NetworkMesh:build_mesh")
    def _build_mesh(self, graph, N, color_strategy, comm, graph_rank):
        if N < 1:
            raise ValueError("N (cells per edge) must be >= 1")
        self._N = int(N)
        if isinstance(graph, ArrayGraph):
            pos = np.asarray(graph.pos, dtype=np.float64)
            edges = np.asarray(graph.edges, dtype=np.int64).reshape(-1, 2)
            in_edge_order = None
        else:
            nodes = np.fromiter(graph.nodes(), dtype=np.int64, count=graph.number_of_nodes())
            if not np.array_equal(nodes, np.arange(nodes.size)):
                raise ValueError("graph nodes must be the integers 0..n-1 in insertion order (mesh.py:183-184,274)")
            pos = np.asarray([graph.nodes[v]["pos"] for v in graph.nodes()], dtype=np.float64)
            edges = _edge_array(graph)
            # graph.in_edges(b) iterates predecessors in insertion order (mesh.py:194)
            in_edge_order = np.asarray(list(graph.in_edges()), dtype=np.int64).reshape(-1, 2)
        if edges.shape[0] == 0:
            raise ValueError("graph has no edges")
        if pos.ndim != 2 or pos.shape[1] not in (1, 2, 3):
            raise ValueError("node positions must have 1, 2 or 3 components")
        n_nodes = pos.shape[0]
        if n_nodes < 2:
            raise ValueError("graph needs at least two nodes")
        if edges.min() < 0 or edges.max() >= n_nodes or np.any(edges[:, 0] == edges[:, 1]):
            raise ValueError("edges must join two distinct existing nodes")
        E = edges.shape[0]
        u, v = edges[:, 0], edges[:, 1]
        self._geom_dim = int(pos.shape[1])  # len(graph.nodes[1]["pos"]), mesh.py:177
        self._node_pos = pos
        self._edges = edges
        self._n_nodes = n_nodes

        colors = _edge_colors(graph, color_strategy, edges)
        self._edge_colors = colors
        self._num_edge_colors = int(np.unique(colors).size)  # mesh.py:179
        if colors.min() < 0 or colors.max() != self._num_edge_colors - 1:
            raise ValueError("edge colours must be 0..C-1")

        # degrees, bifurcations, boundary nodes (mesh.py:182-187)
        deg_in = np.bincount(v, minlength=n_nodes)
        deg_out = np.bincount(u, minlength=n_nodes)
        degree = deg_in + deg_out
        if self._node_degree_override is not None:
            degree = np.asarray(self._node_degree_override, dtype=np.int64)
            if degree.shape != (n_nodes,) or np.any(degree < deg_in + deg_out):
                raise ValueError("node_degree must give the global degree (>= local degree) of every node")
        self._degree = degree
        self._bifurcation_values = np.flatnonzero(degree > 1)
        self._boundary_values = np.flatnonzero(degree == 1)
        self._max_connections = int(degree.max())
        lm = np.full(n_nodes, -1, dtype=np.int32)
        lm[self._bifurcation_values] = np.arange(self._bifurcation_values.size, dtype=np.int32)
        self._node_lm = lm
        n_bif = self._bifurcation_values.size

        # in/out edge colours of every bifurcation (mesh.py:189-209): out-edges in adjacency order
        # (= graph.edges() order), in-edges in predecessor-insertion order
        out_sel = np.flatnonzero(lm[u] >= 0)
        out_sel = out_sel[np.argsort(lm[u[out_sel]], kind="stable")]
        self._bifurcation_out_color = AdjacencyList(
            colors[out_sel], np.concatenate([[0], np.cumsum(np.bincount(lm[u[out_sel]], minlength=n_bif))])
        )
        if in_edge_order is None:
            in_ids = np.flatnonzero(lm[v] >= 0)
        else:
            key = u * n_nodes + v
            order = np.argsort(key)
            in_ids_all = order[np.searchsorted(key[order], in_edge_order[:, 0] * n_nodes + in_edge_order[:, 1])]
            in_ids = in_ids_all[lm[v[in_ids_all]] >= 0]
        in_ids = in_ids[np.argsort(lm[v[in_ids]], kind="stable")]
        self._bifurcation_in_color = AdjacencyList(
            colors[in_ids], np.concatenate([[0], np.cumsum(np.bincount(lm[v[in_ids]], minlength=n_bif))])
        )

        # boundary nodes: with an in-edge -> in_marker (outlet), with an out-edge -> out_marker
        # (inlet)  (mesh.py:211-225, 402-408)
        bnd = self._boundary_values
        self._boundary_in_nodes = bnd[deg_in[bnd] == 1].astype(np.int32)
        self._boundary_out_nodes = bnd[deg_out[bnd] == 1].astype(np.int32)
        self._in_marker = 3 * n_nodes
        self._out_marker = 5 * n_nodes

        # flux slots: colour blocks in order, edges of one colour in ascending edge order
        order = np.argsort(colors, kind="stable")
        slot = np.empty(E, dtype=np.int32)
        slot[order] = np.arange(E, dtype=np.int32)
        self._edge_slot = slot
        self._color_count = np.bincount(colors, minlength=self._num_edge_colors)
        self._color_edges_order = order  # edges sorted by (colour, edge id)
        self._color_start = np.concatenate([[0], np.cumsum(self._color_count)])

        # incidences of every bifurcation sorted by flux slot: 2*e+1 in-edge, 2*e out-edge
        e_in = np.flatnonzero(lm[v] >= 0)
        e_out = np.flatnonzero(lm[u] >= 0)
        inc_lm = np.concatenate([lm[v[e_in]], lm[u[e_out]]])
        inc_code = np.concatenate([2 * e_in + 1, 2 * e_out]).astype(np.int32)
        inc_slot = np.concatenate([slot[e_in], slot[e_out]])
        srt = np.lexsort((inc_slot, inc_lm))
        self._bif_inc = np.ascontiguousarray(inc_code[srt])
        self._bif_ptr = np.concatenate([[0], np.cumsum(np.bincount(inc_lm, minlength=n_bif))]).astype(np.int32)

        n_cells = self._N * E
        n_vertices = n_nodes + (self._N - 1) * E
        self._n_cells, self._n_vertices = n_cells, n_vertices
        self._msh = Mesh(
            self._comm,
            Topology(1, {0: n_vertices, 1: n_cells}, self._cells),
            Geometry(self._geom_dim, self._geometry_x),
            name="network_mesh",
        )
        # cell tags = colour (mesh.py:353-363); vertex tags (mesh.py:402-420)
        self._subdomains = None
        self._facet_markers = None
        self._orientation = OrientationFunction(n_cells, self._cells)

    # ---- device -----------------------------------------------------------------------------
    @property
    def device(self) -> Device:
        """The CUDA context holding this network (created on first use; raises without a GPU)."""
        if self._dev is None:
            d = self._device_arg
            # each NetworkMesh owns its ctx (a ctx holds one network)
            dev = Device(d.index if isinstance(d, Device) else (0 if d is None else int(d)))
            pos = np.ascontiguousarray(self._node_pos, dtype=np.float64)
            eu = np.ascontiguousarray(self._edges[:, 0], dtype=np.int32)
            ev = np.ascontiguousarray(self._edges[:, 1], dtype=np.int32)
            dev.call(
                "nxfx_set_network",
                self._n_nodes, self._edges.shape[0], self._geom_dim, self._N,
                _lib.as_f64p(pos), _lib.as_i32p(eu), _lib.as_i32p(ev), _lib.as_i32p(self._edge_slot),
                _lib.as_i32p(self._node_lm), self._bifurcation_values.size,
                _lib.as_i32p(self._bif_ptr), _lib.as_i32p(self._bif_inc),
            )
            self._dev = dev
        return self._dev

    def geometry_device(self) -> DeviceArray:
        """Borrowed view of the device vertex records {x, y, z, p_bc}, shape (n_vertices*4,)."""
        p = C.c_void_p()
        self.device.call("nxfx_mesh_geometry_device", C.byref(p))
        return DeviceArray(self.device, self._n_vertices * 4, np.float64, ptr=p.value)

    def vertex_coordinates_device(self):
        """The vertex coordinates on the GPU: a ``(n_vertices, 3)`` float64 CUDA ``torch.Tensor`` viewing the
        32-byte vertex records of the device (row stride 4), without a copy -- for evaluating ``p_bc(x, t)`` on the
        GPU and handing it to :meth:`HydraulicNetworkAssembler.compute_forms`.  The view is borrowed from the
        context (valid while this mesh lives) and is READ-ONLY by contract: the assembly reads the cell lengths
        from these records, and torch has no read-only tensors (it refuses the read-only flag of
        ``__cuda_array_interface__``), so nothing stops a write.  Work enqueued on the current torch stream after
        this call sees the coordinates the library has enqueued so far."""
        p = C.c_void_p()
        dev = self.device
        dev.call("nxfx_mesh_geometry_device", C.byref(p))
        nv = self._n_vertices
        view = DeviceArray(dev, nv * 4, np.float64, ptr=p.value, shape=(nv, 3), strides=(32, 8))
        view._owner = self  # the records belong to this mesh's context
        dev.torch_wait()
        return view.as_tensor()

    def _geometry_x(self) -> npt.NDArray[np.float64]:
        if self._x_host is None:
            self._x_host = np.ascontiguousarray(self.geometry_device().download().reshape(-1, 4)[:, :3])
        return self._x_host

    def _cells(self) -> npt.NDArray[np.int64]:
        """Cell -> vertex table (mesh.py:293-309), built on demand."""
        if self._cells_host is None:
            E, N = self._edges.shape[0], self._N
            chain = np.empty((E, N + 1), dtype=np.int64)
            chain[:, 0] = self._edges[:, 0]
            chain[:, N] = self._edges[:, 1]
            if N > 1:
                chain[:, 1:N] = self._n_nodes + np.arange(E)[:, None] * (N - 1) + np.arange(N - 1)[None, :]
            self._cells_host = np.stack([chain[:, :-1].ravel(), chain[:, 1:].ravel()], axis=1)
        return self._cells_host

    # ---- submeshes --------------------------------------------------------------------------
    @timed("nxfx:NetworkMesh:build_network_submeshes")
    def _build_network_submeshes(self):
        """One submesh per colour (mesh.py:425-460), materialised lazily."""
        C_ = self._num_edge_colors
        self._edge_meshes = _LazyList(C_, self._make_submesh)
        self._edge_entity_maps = _LazyList(C_, self._make_entity_map)
        self._submesh_facet_markers = _LazyList(C_, self._make_submesh_facet_markers)

    def color_edges(self, color: int) -> npt.NDArray[np.int64]:
        """Graph edges of a colour in ascending order."""
        s, e = self._color_start[color], self._color_start[color + 1]
        return self._color_edges_order[s:e]

    def _submesh_vertices(self, color: int) -> npt.NDArray[np.int64]:
        """Parent vertices of the colour submesh, sorted (create_submesh keeps parent order)."""
        edges = self.color_edges(color)
        N = self._N
        ends = self._edges[edges].ravel()
        if N > 1:
            inner = (self._n_nodes + edges[:, None] * (N - 1) + np.arange(N - 1)[None, :]).ravel()
            return np.unique(np.concatenate([ends, inner]))
        return np.unique(ends)

    def _make_entity_map(self, color: int) -> EntityMap:
        edges = self.color_edges(color)
        cells = (edges[:, None] * self._N + np.arange(self._N)[None, :]).ravel()
        return EntityMap(cells, self._n_cells)

    def _make_submesh(self, color: int) -> Mesh:
        edges = self.color_edges(color)
        verts = self._submesh_vertices(color)
        nm = self

        def sub_x():
            return nm._geometry_x()[verts]

        def sub_cells():
            parent_cells = nm._cells()[nm._make_entity_map(color).sub_topology_to_topology(
                np.arange(edges.size * nm._N, dtype=np.int32))]
            return np.searchsorted(verts, parent_cells)

        m = Mesh(
            self._comm,
            Topology(1, {0: verts.size, 1: edges.size * self._N}, sub_cells),
            Geometry(self._geom_dim, sub_x),
            name=f"submesh_{color}",
        )
        m.parent_vertices = verts
        return m

    def _make_submesh_facet_markers(self, color: int) -> MeshTags:
        verts = self._submesh_vertices(color)
        tags = self.boundaries
        marker = np.full(self._n_vertices, -1, dtype=np.int32)
        marker[tags.indices] = tags.values
        vals = marker[verts]
        sel = np.flatnonzero(vals >= 0)
        return MeshTags(self.submeshes[color], 0, sel, vals[sel].copy())

    @timed("nxfx:NetworkMesh:create_lm_submesh")
    def _create_lm_submesh(self):
        """Point-cloud submesh of the bifurcation vertices (mesh.py:117-136)."""
        bif = self._bifurcation_values
        nm = self
        self._lm_mesh = Mesh(
            self._comm,
            Topology(0, {0: bif.size}),
            Geometry(self._geom_dim, lambda: nm._geometry_x()[bif]),
            name="lm_mesh",
        )
        self._lm_map = EntityMap(bif, self._n_vertices)

    # ---- reference accessors (mesh.py:98-115, 462-538) ---------------------------------------
    @property
    def lm_mesh(self) -> Mesh:
        """Lagrange multiplier mesh, a point-cloud mesh including each bifurcation."""
        return self._lm_mesh

    @property
    def lm_map(self) -> EntityMap:
        return self._lm_map

    @property
    def comm(self):
        return self.mesh.comm

    @property
    def submesh_facet_markers(self):
        return self._submesh_facet_markers

    @property
    def mesh(self) -> Mesh:
        return self._msh

    @property
    def subdomains(self) -> MeshTags:
        """Cell tags: colour of the graph edge the cell belongs to (mesh.py:353-363)."""
        if self._subdomains is None:
            self._subdomains = MeshTags(
                self._msh, 1, np.arange(self._n_cells, dtype=np.int32),
                np.repeat(self._edge_colors, self._N).astype(np.int32), name="subdomains",
            )
        return self._subdomains

    @property
    def boundaries(self) -> MeshTags:
        """Vertex tags of the graph nodes: node id, ``in_marker`` on outlets, ``out_marker`` on
        inlets (mesh.py:402-420)."""
        if self._facet_markers is None:
            vals = np.arange(self._n_nodes, dtype=np.int32)
            vals[self._boundary_in_nodes] = self._in_marker
            vals[self._boundary_out_nodes] = self._out_marker
            self._facet_markers = MeshTags(
                self._msh, 0, np.arange(self._n_nodes, dtype=np.int32), vals, name="bifurcations"
            )
        return self._facet_markers

    @property
    def submeshes(self):
        return self._edge_meshes

    @property
    def entity_maps(self):
        return self._edge_entity_maps

    @property
    def orientation(self) -> OrientationFunction:
        """DG-0 field containing the orientation of the tangent vector of the graph."""
        return self._orientation

    @property
    def bifurcation_values(self) -> npt.NDArray[np.int32]:
        return self._bifurcation_values

    @property
    def boundary_values(self) -> npt.NDArray[np.int32]:
        return self._boundary_values

    def in_edges(self, bifurcation_idx: int) -> npt.NDArray[np.int32]:
        """Colours of the in-edges of bifurcation ``bifurcation_idx`` (index into
        ``bifurcation_values``)."""
        assert bifurcation_idx < len(self.bifurcation_values)
        return self._bifurcation_in_color.links(np.int32(bifurcation_idx))

    def out_edges(self, bifurcation_idx: int) -> npt.NDArray[np.int32]:
        assert bifurcation_idx < len(self.bifurcation_values)
        return self._bifurcation_out_color.links(np.int32(bifurcation_idx))

    @property
    def num_edge_colors(self) -> int:
        return self._num_edge_colors

    @property
    def in_marker(self) -> int:
        return self._in_marker

    @property
    def out_marker(self) -> int:
        return self._out_marker

    # ---- extensions used by the assembler / solver -------------------------------------------
    @property
    def cells_per_edge(self) -> int:
        return self._N

    @property
    def graph_edges(self) -> npt.NDArray[np.int64]:
        return self._edges

    @property
    def edge_colors(self) -> npt.NDArray[np.int32]:
        return self._edge_colors

    @property
    def edge_slot(self) -> npt.NDArray[np.int32]:
        return self._edge_slot

    @property
    def node_multiplier_index(self) -> npt.NDArray[np.int32]:
        return self._node_lm

    def oriented_tangent_integral(self, direction) -> float:
        """``assemble_scalar(inner(direction, t) * orientation * dx)`` on the device-generated
        vertices (tests/test_orientation.py:45-50 re-expressed without UFL)."""
        x = self._geometry_x()
        cells = self._cells()
        d = np.zeros(3)
        d[: len(direction)] = direction
        return float(np.sum(((x[cells[:, 1]] - x[cells[:, 0]]) @ d) * self.orientation.x.array))
