"""NumPy/SciPy restatement of the networks_fenicsx assemble-and-solve hot path (CPU oracle).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  All ``file:line`` citations point into
the upstream reference tree (``src/networks_fenicsx/...``).  The reference delegates all
arithmetic to DOLFINx/FFCx/PETSc/MUMPS, none of which can be installed in this image, so the
assembled values and the solution are **parity unpinned** by the reference itself; they are pinned
by the closed-form resistor-network answer (``resistor_network_solution``) and the known-answer
values in ``tests/test_oracle_kat.py``.  Everything structural (graph analysis, colouring, mesh
arrays, orientation, block order) is pinned by the reference's own tests and by fixtures generated
from the reference's ``network_generation.py`` (``tests/golden/make_golden.py``).

Two layers:

* ``*_literal`` functions follow the reference's per-edge / per-bifurcation Python loops one to one
  (small cases only);
* ``OracleNetwork`` is the vectorised form used at benchmark sizes; the tests check it against the
  literal layer.

Numbering is the canonical serial numbering of SURVEY.md Appendix C: cells ``e*N + j`` in
``graph.edges()`` order, vertices in input order, flux dofs per colour block in ascending edge
order, pressure dof = cell id, multiplier dof = index into ``bifurcation_values``; global order
``[q_0 .. q_{C-1}, p, lambda]`` (assembly.py:318-321).
"""

from __future__ import annotations

import dataclasses

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

THIRD = 1.0 / 3.0
SIXTH = 1.0 / 6.0


# --------------------------------------------------------------------------------------
# Literal layer (loops; follows the reference statement by statement)
# --------------------------------------------------------------------------------------
def color_graph_literal(graph, strategy):
    """Edge colouring, mesh.py:29-42.

    ``strategy is None``: colour = position of the edge in ``graph.edges`` (mesh.py:41).
    Otherwise greedy colouring of the line graph of the undirected graph (mesh.py:38-39).
    """
    import networkx as nx

    if strategy is None:
        return {edge: i for i, edge in enumerate(graph.edges)}
    line = nx.line_graph(graph.to_undirected())
    return nx.coloring.greedy_color(line, strategy=strategy)


def lookup_color(coloring, u, v):
    """Orientation-insensitive lookup (the reference indexes ``coloring[(u, v)]``, mesh.py:282,313;
    networkx may key an undirected line-graph node as ``(v, u)`` -- SURVEY Appendix D)."""
    key = (u, v)
    if key in coloring:
        return coloring[key]
    return coloring[(v, u)]


@dataclasses.dataclass
class GraphInfo:
    geom_dim: int
    num_edge_colors: int
    number_of_nodes: int
    max_connections: int
    bifurcation_values: np.ndarray
    boundary_values: np.ndarray
    in_color: np.ndarray
    in_offsets: np.ndarray
    out_color: np.ndarray
    out_offsets: np.ndarray
    boundary_in_nodes: np.ndarray  # nodes with one in-edge  (outlets, tagged in_marker)
    boundary_out_nodes: np.ndarray  # nodes with one out-edge (inlets,  tagged out_marker)


def analyse_graph_literal(graph, coloring) -> GraphInfo:
    """Graph analysis on the rank that holds the graph, mesh.py:175-225."""
    n_nodes = graph.number_of_nodes()
    deg = np.full(n_nodes, -1, dtype=np.int32)
    for node, d in graph.degree():
        deg[node] = d
    bif = np.flatnonzero(deg > 1)
    bnd = np.flatnonzero(deg == 1)
    in_c, in_o, out_c, out_o = [], [0], [], [0]
    for b in bif:
        for e in graph.in_edges(b):
            in_c.append(lookup_color(coloring, *e))
        in_o.append(len(in_c))
        for e in graph.out_edges(b):
            out_c.append(lookup_color(coloring, *e))
        out_o.append(len(out_c))
    b_in, b_out = [], []
    for b in bnd:
        n_in, n_out = len(graph.in_edges(b)), len(graph.out_edges(b))
        assert n_in + n_out == 1
        (b_in if n_in == 1 else b_out).append(b)
    return GraphInfo(
        geom_dim=len(graph.nodes[1]["pos"]),
        num_edge_colors=len(set(coloring.values())),
        number_of_nodes=n_nodes,
        max_connections=int(deg.max()),
        bifurcation_values=bif,
        boundary_values=bnd,
        in_color=np.asarray(in_c, dtype=np.int32),
        in_offsets=np.asarray(in_o, dtype=np.int32),
        out_color=np.asarray(out_c, dtype=np.int32),
        out_offsets=np.asarray(out_o, dtype=np.int32),
        boundary_in_nodes=np.asarray(b_in, dtype=np.int32),
        boundary_out_nodes=np.asarray(b_out, dtype=np.int32),
    )


def mesh_arrays_literal(graph, N, coloring):
    """Mesh nodes / cells / markers / input orientation, mesh.py:270-324.

    Nodes: graph nodes in ``graph.nodes()`` order, then for each edge (``graph.edges()`` order) its
    ``N-1`` interior points ``start*(1-w) + end*w`` with ``w = linspace(0,1,N,endpoint=False)[1:]``.
    Cells of an edge run from ``u`` to ``v``.  Orientation input: ``+1`` iff ``cell[0] < cell[1]``.
    """
    coords = np.asarray([graph.nodes[v]["pos"] for v in graph.nodes()], dtype=np.float64)
    w = np.linspace(0, 1, N, endpoint=False)[1:]
    nodes = [row for row in coords]
    cells, markers = [], []
    for u, v in graph.edges():
        col = lookup_color(coloring, u, v)
        first_new = len(nodes)
        for wk in w:
            nodes.append(coords[u] * (1 - wk) + coords[v] * wk)
        chain = [u] + list(range(first_new, first_new + len(w))) + [v]
        for a, b in zip(chain[:-1], chain[1:]):
            cells.append((a, b))
            markers.append(col)
    cells_ = np.asarray(cells, dtype=np.int64).reshape(-1, 2)
    markers_ = np.asarray(markers, dtype=np.int32)
    orient = np.where(cells_[:, 0] < cells_[:, 1], 1.0, -1.0)
    return np.asarray(nodes, dtype=np.float64), cells_, markers_, orient


def orientation_net_effect(cells):
    """Net DG0 orientation after the reorder correction, mesh.py:365-400.

    The input sign (mesh.py:321-322) is flipped wherever the created cell's geometry nodes are not
    ascending in input index (mesh.py:379-398); interval cells keep their node order, so the
    product is +1 on every cell and ``orientation * t`` is the unit tangent u->v (SURVEY A.2).
    """
    s_in = np.where(cells[:, 0] < cells[:, 1], 1.0, -1.0)
    in_order = cells[:, 0] < cells[:, 1]
    return np.where(in_order, s_in, -s_in)


def vertex_markers_literal(info: GraphInfo):
    """Vertex tags of the graph nodes, mesh.py:402-408."""
    in_marker = 3 * info.number_of_nodes
    out_marker = 5 * info.number_of_nodes
    tags = np.arange(info.number_of_nodes, dtype=np.int32)
    tags[info.boundary_in_nodes] = in_marker
    tags[info.boundary_out_nodes] = out_marker
    return tags, in_marker, out_marker


def integration_entities_literal(graph, N, coloring, info: GraphInfo):
    """(parent cell, local facet) pairs per colour, assembly.py:28-92, in closed form: an edge
    (u, v) entering bifurcation v contributes (last cell of the edge, facet 1) to the influx list of
    its colour; an edge leaving bifurcation u contributes (first cell, facet 0) to the outflux list.
    Pairs are listed in ascending parent cell order (the submesh keeps parent order)."""
    bif = set(int(b) for b in info.bifurcation_values)
    infl = {c: [] for c in range(info.num_edge_colors)}
    outfl = {c: [] for c in range(info.num_edge_colors)}
    for e, (u, v) in enumerate(graph.edges()):
        c = lookup_color(coloring, u, v)
        if u in bif:
            outfl[c] += [e * N, 0]
        if v in bif:
            infl[c] += [e * N + N - 1, 1]
    as_arr = lambda d: {c: np.asarray(x, dtype=np.int32) for c, x in d.items()}  # noqa: E731
    return as_arr(infl), as_arr(outfl)


def assemble_literal(graph, N, coloring, p_bc, R=1.0, f=0.0):
    """Dense, loop-based assembly of the block system (assembly.py:243-277, 354-367) for small
    graphs.  Returns ``(A_dense, b, stored)`` where ``stored`` is the boolean sparsity pattern
    including the explicit zeros DOLFINx inserts for the multiplier blocks (SURVEY A.3)."""
    info = analyse_graph_literal(graph, coloring)
    nodes, cells, markers, _ = mesh_arrays_literal(graph, N, coloring)
    edges = list(graph.edges())
    C = info.num_edge_colors
    ecol = [lookup_color(coloring, u, v) for u, v in edges]
    rank, count = [], [0] * C
    for c in ecol:
        rank.append(count[c])
        count[c] += 1
    qoff = np.concatenate([[0], np.cumsum([n * (N + 1) for n in count])])
    poff = int(qoff[-1])
    loff = poff + N * len(edges)
    lm_of = {int(b): i for i, b in enumerate(info.bifurcation_values)}
    n = loff + len(lm_of)
    A = np.zeros((n, n))
    stored = np.zeros((n, n), dtype=bool)
    b = np.zeros(n)
    pad = np.zeros((nodes.shape[0], 3))
    pad[:, : nodes.shape[1]] = nodes
    pbc = np.asarray(p_bc(pad.T), dtype=np.float64) * np.ones(nodes.shape[0])

    def add(i, j, val):
        A[i, j] += val
        stored[i, j] = True

    for e, (u, v) in enumerate(edges):
        fb = int(qoff[ecol[e]]) + rank[e] * (N + 1)
        for j in range(N):
            cell = e * N + j
            x0, x1 = pad[cells[cell, 0]], pad[cells[cell, 1]]
            d = x1 - x0
            h = np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
            m = R * h
            q0, q1, pr = fb + j, fb + j + 1, poff + cell
            add(q0, q0, m * THIRD)
            add(q0, q1, m * SIXTH)
            add(q1, q0, m * SIXTH)
            add(q1, q1, m * THIRD)
            add(pr, q0, -1.0)  # a[P][i] = +int phi dq/ds   (assembly.py:254)
            add(pr, q1, +1.0)
            add(q0, pr, +1.0)  # a[i][P] = -int p dv/ds     (assembly.py:255)
            add(q1, pr, -1.0)
            b[pr] += f * h  # L[P] = int f phi            (assembly.py:262)
        if v in lm_of:  # influx: +mu q at the last vertex   (assembly.py:271-273)
            lm = loff + lm_of[v]
            add(lm, fb + N - 1, 0.0)
            add(lm, fb + N, 1.0)
            add(fb + N - 1, lm, 0.0)
            add(fb + N, lm, 1.0)
        else:  # outlet boundary vertex: +p_bc v        (assembly.py:258)
            b[fb + N] += pbc[v]
        if u in lm_of:  # outflux: -mu q at the first vertex  (assembly.py:275-277)
            lm = loff + lm_of[u]
            add(lm, fb, -1.0)
            add(lm, fb + 1, 0.0)
            add(fb, lm, -1.0)
            add(fb + 1, lm, 0.0)
        else:  # inlet boundary vertex: -p_bc v         (assembly.py:258-260)
            b[fb] -= pbc[u]
    return A, b, stored


# --------------------------------------------------------------------------------------
# Vectorised layer
# --------------------------------------------------------------------------------------
def graph_to_arrays(graph, coloring):
    """``(pos[n_nodes,gdim], edges[E,2], colors[E])`` in ``graph.nodes()`` / ``graph.edges()`` order."""
    pos = np.asarray([graph.nodes[v]["pos"] for v in graph.nodes()], dtype=np.float64)
    edges = np.asarray([[u, v] for u, v in graph.edges()], dtype=np.int64).reshape(-1, 2)
    colors = np.asarray([lookup_color(coloring, u, v) for u, v in graph.edges()], dtype=np.int32)
    return pos, edges, colors


class OracleNetwork:
    """Vectorised oracle of mesh arrays, dof tables, pattern, assembly and solve."""

    def __init__(self, pos, edges, colors, N: int, degree=None):
        """``degree``: global node degrees when (pos, edges) is one part of a partitioned network
        (test support for the multi-GPU partition; the reference has no such notion)."""
        pos = np.asarray(pos, dtype=np.float64)
        self.pos = pos
        self.edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
        self.colors = np.asarray(colors, dtype=np.int32)
        self.N = int(N)
        self.n_nodes, self.gdim = pos.shape
        self.E = self.edges.shape[0]
        E, N = self.E, self.N
        u, v = self.edges[:, 0], self.edges[:, 1]
        # mesh.py:182-187
        self.degree = np.bincount(u, minlength=self.n_nodes) + np.bincount(v, minlength=self.n_nodes)
        if degree is not None:
            self.degree = np.asarray(degree)
        self.bifurcation_values = np.flatnonzero(self.degree > 1)
        self.boundary_values = np.flatnonzero(self.degree == 1)
        self.lm_index = np.full(self.n_nodes, -1, dtype=np.int64)
        self.lm_index[self.bifurcation_values] = np.arange(self.bifurcation_values.size)
        self.n_bif = self.bifurcation_values.size
        self.C = int(np.unique(self.colors).size)
        # mesh.py:270-324 (vectorised)
        w = np.linspace(0, 1, N, endpoint=False)[1:]
        inner = pos[u][:, None, :] * (1 - w)[None, :, None] + pos[v][:, None, :] * w[None, :, None]
        self.x = np.vstack([pos, inner.reshape(-1, self.gdim)])
        self.x3 = np.zeros((self.x.shape[0], 3))
        self.x3[:, : self.gdim] = self.x
        chain = np.empty((E, N + 1), dtype=np.int64)
        chain[:, 0] = u
        chain[:, N] = v
        if N > 1:
            chain[:, 1:N] = self.n_nodes + np.arange(E)[:, None] * (N - 1) + np.arange(N - 1)[None, :]
        self.cells = np.stack([chain[:, :-1].ravel(), chain[:, 1:].ravel()], axis=1)
        self.cell_markers = np.repeat(self.colors, N)
        self.orientation = orientation_net_effect(self.cells)
        # dof tables (SURVEY Appendix C)
        order = np.argsort(self.colors, kind="stable")
        count = np.bincount(self.colors, minlength=self.C)
        start = np.concatenate([[0], np.cumsum(count)])
        self.rank = np.empty(E, dtype=np.int64)
        self.rank[order] = np.arange(E) - start[self.colors[order]]
        self.qoff = np.concatenate([[0], np.cumsum(count * (N + 1))])
        self.fb = self.qoff[self.colors] + self.rank * (N + 1)
        self.poff = int(self.qoff[-1])
        self.pb = self.poff + np.arange(E) * N
        self.loff = self.poff + N * E
        self.n_dofs = self.loff + self.n_bif
        self.block_sizes = [int(c) * (N + 1) for c in count] + [N * E, self.n_bif]

    # geometry --------------------------------------------------------------------
    def cell_lengths(self):
        d = self.x3[self.cells[:, 1]] - self.x3[self.cells[:, 0]]
        return np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])

    def oriented_tangent_integral(self, direction):
        """sum_c h_c (direction . t_c) orientation_c  -- tests/test_orientation.py:45-50."""
        d = self.x3[self.cells[:, 1]] - self.x3[self.cells[:, 0]]
        dvec = np.zeros(3)
        dvec[: len(direction)] = direction
        return float(np.sum((d @ dvec) * self.orientation))

    def eval_pbc(self, p_bc):
        """p_bc interpolated into P1 on the parent mesh: nodal values at x (3, npoints) --
        assembly.py:225-234."""
        val = np.asarray(p_bc(self.x3.T), dtype=np.float64)
        return val * np.ones(self.x3.shape[0])

    # assembly --------------------------------------------------------------------
    def assemble(self, pbc_vertex, R=1.0, f=0.0):
        """COO -> CSR assembly of the monolithic block system incl. explicit zeros.

        assembly.py:253-277 (forms), :354-367 (assemble semantics)."""
        E, N = self.E, self.N
        h = self.cell_lengths()
        Rc = np.broadcast_to(np.asarray(R, dtype=np.float64), h.shape)
        fc = np.broadcast_to(np.asarray(f, dtype=np.float64), h.shape)
        m = Rc * h
        j = np.tile(np.arange(N), E)
        e = np.repeat(np.arange(E), N)
        q0 = self.fb[e] + j
        q1 = q0 + 1
        pr = self.poff + np.arange(E * N)
        one = np.ones(E * N)
        rows = [q0, q0, q1, q1, pr, pr, q0, q1]
        cols = [q0, q1, q0, q1, q0, q1, pr, pr]
        vals = [m * THIRD, m * SIXTH, m * SIXTH, m * THIRD, -one, one, one, -one]
        u, v = self.edges[:, 0], self.edges[:, 1]
        ein = np.flatnonzero(self.lm_index[v] >= 0)  # edge enters bifurcation v
        eout = np.flatnonzero(self.lm_index[u] >= 0)  # edge leaves bifurcation u
        lin = self.loff + self.lm_index[v[ein]]
        lout = self.loff + self.lm_index[u[eout]]
        fin, fout = self.fb[ein], self.fb[eout]
        zi, zo = np.zeros(ein.size), np.zeros(eout.size)
        rows += [lin, lin, fin + N - 1, fin + N, lout, lout, fout, fout + 1]
        cols += [fin + N - 1, fin + N, lin, lin, fout, fout + 1, lout, lout]
        vals += [zi, zi + 1.0, zi, zi + 1.0, zo - 1.0, zo, zo - 1.0, zo]
        A = sp.coo_matrix(
            (np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
            shape=(self.n_dofs, self.n_dofs),
        ).tocsr()
        A.sort_indices()
        b = np.zeros(self.n_dofs)
        b[pr] = fc * h
        outlet = np.flatnonzero(self.lm_index[v] < 0)
        inlet = np.flatnonzero(self.lm_index[u] < 0)
        np.add.at(b, self.fb[outlet] + N, pbc_vertex[v[outlet]])
        np.add.at(b, self.fb[inlet], -pbc_vertex[u[inlet]])
        return A, b

    def expected_nnz(self):
        """nnz = E(7N+1) + 4I, I = 2E - n_boundary (SURVEY Appendix B)."""
        inc = 2 * self.E - self.boundary_values.size
        return self.E * (7 * self.N + 1) + 4 * inc

    @staticmethod
    def solve(A, b):
        """Direct solve (SuperLU as the MUMPS stand-in) -- solver.py:58-65,127."""
        return spla.splu(A.tocsc()).solve(b)

    @staticmethod
    def solve_exact(A, r, rounds=4):
        """``A^{-1} r`` to well below float64 rounding, as ``np.longdouble`` (test reference for operators that are
        meant to be exact solves).  SuperLU in float64, then ``rounds`` steps of iterative refinement whose residual
        ``r - A x`` is formed in extended precision (x86 long double: 64-bit mantissa, eps 1.1e-19).  Each step gains
        about -log10(eps_64 cond(A)) digits until the extended residual's own rounding is reached.  ``r`` may be
        ``[n]`` or ``[n, k]``."""
        lu = spla.splu(sp.csc_matrix(A, dtype=np.float64))
        Ald = sp.csr_matrix(A).astype(np.longdouble)
        rld = np.asarray(r).astype(np.longdouble)
        x = lu.solve(np.asarray(r, dtype=np.float64)).astype(np.longdouble)
        for _ in range(rounds):
            res = rld - Ald @ x
            x += lu.solve(res.astype(np.float64))
        return x

    @staticmethod
    def gmres_reference(A, b, minv_diag, m, k_max):
        """Right-preconditioned GMRES(m) from x0 = 0 in ``np.longdouble``: Arnoldi with modified Gram-Schmidt and
        one re-orthogonalisation, Givens rotations.  ``minv_diag``: the preconditioner as a diagonal (None: the
        identity).  Returns ``(rho, beta, x)``: ``rho[k]`` the minimal residual norm after k iterations (k = 0 ..
        k_max; within a cycle the least-squares residual, at a restart the true residual of the updated iterate),
        ``beta[c]`` the true residual norm at the start of cycle c (one more entry after the last cycle), and the
        final iterate."""
        ld = np.longdouble
        n = b.size
        Ald = sp.csr_matrix(A).astype(ld)
        bl = np.asarray(b).astype(ld)
        dinv = np.ones(n, dtype=ld) if minv_diag is None else np.asarray(minv_diag).astype(ld)
        x = np.zeros(n, dtype=ld)
        rho, beta = [], []
        its = 0
        while True:
            r = bl - Ald @ x
            bt = np.sqrt(np.sum(r * r))
            beta.append(bt)
            if its == 0:
                rho.append(bt)
            else:
                rho[-1] = bt  # the true residual of the restarted iterate replaces the estimate
            if its >= k_max or bt == 0:
                break
            V = np.zeros((m + 1, n), dtype=ld)
            H = np.zeros((m + 1, m), dtype=ld)
            cs, sn = np.zeros(m, dtype=ld), np.zeros(m, dtype=ld)
            g = np.zeros(m + 1, dtype=ld)
            g[0] = bt
            V[0] = r / bt
            k = 0
            while k < m and its < k_max:
                w = Ald @ (dinv * V[k])
                for _ in range(2):  # MGS, then once more
                    for i in range(k + 1):
                        h = np.sum(V[i] * w)
                        H[i, k] += h
                        w -= h * V[i]
                H[k + 1, k] = np.sqrt(np.sum(w * w))
                breakdown = not H[k + 1, k] > 0  # the Krylov space is invariant: the iterate below is exact
                if not breakdown:
                    V[k + 1] = w / H[k + 1, k]
                for i in range(k):
                    t = cs[i] * H[i, k] + sn[i] * H[i + 1, k]
                    H[i + 1, k] = -sn[i] * H[i, k] + cs[i] * H[i + 1, k]
                    H[i, k] = t
                den = np.hypot(H[k, k], H[k + 1, k])
                cs[k], sn[k] = (H[k, k] / den, H[k + 1, k] / den) if den > 0 else (ld(1), ld(0))
                H[k, k] = den
                g[k + 1] = -sn[k] * g[k]
                g[k] = cs[k] * g[k]
                rho.append(abs(g[k + 1]))
                k += 1
                its += 1
                if breakdown:
                    break
            y = np.zeros(k, dtype=ld)
            for i in range(k - 1, -1, -1):
                y[i] = (g[i] - H[i, i + 1:k] @ y[i + 1:]) / H[i, i]
            x += dinv * (V[:k].T @ y)
        return np.asarray(rho, dtype=ld), np.asarray(beta, dtype=ld), x

    def split(self, x):
        """Split the blocked vector as fem.petsc.assign does -- solver.py:120-134."""
        bounds = np.concatenate([[0], np.cumsum(self.block_sizes)])
        return [x[bounds[i] : bounds[i + 1]] for i in range(len(self.block_sizes))]

    def global_flux(self, x):
        """DG1 global flux on the parent mesh, post_processing.py:19-52: per cell the two flux
        values of its edge dofs; dof 2*cell + local."""
        E, N = self.E, self.N
        j = np.tile(np.arange(N), E)
        e = np.repeat(np.arange(E), N)
        q0 = self.fb[e] + j
        return np.stack([x[q0], x[q0 + 1]], axis=1).ravel()

    # closed-form known answer ----------------------------------------------------
    def resistor_network_solution(self, pbc_vertex, R=1.0):
        """Closed form for f = 0 (SURVEY A.3): resistor network on the bifurcation nodes with
        boundary pressures -p_bc.  Returns (q_edge[E], lambda[n_bif])."""
        E, N = self.E, self.N
        h = self.cell_lengths().reshape(E, N)
        Rc = np.broadcast_to(np.asarray(R, dtype=np.float64), (E * N,)).reshape(E, N)
        g = 1.0 / np.sum(Rc * h, axis=1)
        u, v = self.edges[:, 0], self.edges[:, 1]
        lu, lv = self.lm_index[u], self.lm_index[v]
        nb = self.n_bif
        L = sp.lil_matrix((nb, nb))
        rhs = np.zeros(nb)
        for k in range(E):
            a, c = lu[k], lv[k]
            if a >= 0:
                L[a, a] += g[k]
            if c >= 0:
                L[c, c] += g[k]
            if a >= 0 and c >= 0:
                L[a, c] -= g[k]
                L[c, a] -= g[k]
            if a < 0 and c >= 0:  # inlet edge, boundary pressure -p_bc(x_u)
                rhs[c] += g[k] * (-pbc_vertex[u[k]])
            if c < 0 and a >= 0:  # outlet edge, boundary pressure -p_bc(x_v)
                rhs[a] += g[k] * (-pbc_vertex[v[k]])
        lam = spla.spsolve(L.tocsc(), rhs) if nb else np.zeros(0)
        lam = np.atleast_1d(lam)
        pu = np.where(lu >= 0, lam[np.maximum(lu, 0)] if nb else 0.0, -pbc_vertex[u])
        pv = np.where(lv >= 0, lam[np.maximum(lv, 0)] if nb else 0.0, -pbc_vertex[v])
        return g * (pu - pv), lam


# --------------------------------------------------------------------------------------
# Higher-order elements: flux P_fd (continuous per edge), pressure DG0 (pd = 0) or continuous
# P_pd on the parent mesh (pd >= 1) -- assembly.py:127-146.  Equispaced Lagrange, dof order on a
# cell [X=0, X=1, interior ascending] (basix "equispaced" variant; interval cells need no
# permutations).  Literal COO assembly; canonical numbering (SURVEY Appendix C): flux dofs of an
# edge = [N+1 vertex dofs, then fd-1 interior dofs per cell], pressure dofs = [mesh vertices, then
# pd-1 interior dofs per cell].
# --------------------------------------------------------------------------------------
def lagrange_nodes(d):
    if d == 0:
        return np.array([0.5])
    return np.concatenate([[0.0, 1.0], np.arange(1, d) / d])


def lagrange_tables(fd, pd):
    """(M_ref[fd+1,fd+1], B_ref[pd+1,fd+1], w_ref[pd+1], trace0[fd+1], trace1[fd+1]) by exact
    Gauss-Legendre quadrature: M = int phi_a phi_b, B = int psi_r phi_a', w = int psi_r
    (SURVEY A.3)."""
    from numpy.polynomial import polynomial as P

    def basis(d):
        x = lagrange_nodes(d)
        if d == 0:
            return [np.array([1.0])]
        out = []
        for i in range(d + 1):
            c = np.array([1.0])
            for j in range(d + 1):
                if j != i:
                    c = P.polymul(c, np.array([-x[j], 1.0]) / (x[i] - x[j]))
            out.append(c)
        return out

    phi, psi = basis(fd), basis(pd)
    gx, gw = np.polynomial.legendre.leggauss(fd + pd + 2)
    X, W = 0.5 * (gx + 1.0), 0.5 * gw
    ph = np.array([P.polyval(X, c) for c in phi])
    dph = np.array([P.polyval(X, P.polyder(c)) if c.size > 1 else 0 * X for c in phi])
    ps = np.array([P.polyval(X, c) for c in psi])
    M = (ph * W) @ ph.T
    B = (ps * W) @ dph.T
    w = ps @ W
    t0 = np.array([P.polyval(0.0, c) for c in phi])
    t1 = np.array([P.polyval(1.0, c) for c in phi])
    return M, B, w, np.round(t0), np.round(t1)


class OracleNetworkHO(OracleNetwork):
    """Higher-order oracle (small / medium cases; loop-free COO but not tuned)."""

    def __init__(self, pos, edges, colors, N, flux_degree, pressure_degree):
        super().__init__(pos, edges, colors, N)
        fd, pd = int(flux_degree), int(pressure_degree)
        self.fd, self.pd = fd, pd
        E, N = self.E, self.N
        count = np.bincount(self.colors, minlength=self.C)
        per_edge = fd * N + 1
        self.qoff = np.concatenate([[0], np.cumsum(count * per_edge)])
        self.fb = self.qoff[self.colors] + self.rank * per_edge
        self.poff = int(self.qoff[-1])
        nv = self.x.shape[0]
        self.n_p = N * E if pd == 0 else nv + (pd - 1) * N * E
        self.loff = self.poff + self.n_p
        self.n_dofs = self.loff + self.n_bif
        self.block_sizes = [int(c) * per_edge for c in count] + [self.n_p, self.n_bif]
        self.tables = lagrange_tables(fd, pd)

    def cell_flux_dofs(self):
        """[n_cells, fd+1] global flux dofs: [vertex j, vertex j+1, interior...]."""
        E, N, fd = self.E, self.N, self.fd
        e = np.repeat(np.arange(E), N)
        j = np.tile(np.arange(N), E)
        cols = [self.fb[e] + j, self.fb[e] + j + 1]
        for i in range(fd - 1):
            cols.append(self.fb[e] + (N + 1) + j * (fd - 1) + i)
        return np.stack(cols, axis=1)

    def cell_pressure_dofs(self):
        E, N, pd = self.E, self.N, self.pd
        nc = E * N
        if pd == 0:
            return self.poff + np.arange(nc)[:, None]
        nv = self.x.shape[0]
        cols = [self.poff + self.cells[:, 0], self.poff + self.cells[:, 1]]
        for i in range(pd - 1):
            cols.append(self.poff + nv + np.arange(nc) * (pd - 1) + i)
        return np.stack(cols, axis=1)

    def assemble(self, pbc_vertex, R=1.0, f=0.0):
        M, B, w, t0, t1 = self.tables
        E, N, fd, pd = self.E, self.N, self.fd, self.pd
        h = self.cell_lengths()
        nc = h.size
        Rc = np.broadcast_to(np.asarray(R, dtype=np.float64), h.shape)
        fc = np.broadcast_to(np.asarray(f, dtype=np.float64), h.shape)
        m = Rc * h
        qd, pdofs = self.cell_flux_dofs(), self.cell_pressure_dofs()
        rows, cols, vals = [], [], []
        for a in range(fd + 1):
            for b_ in range(fd + 1):
                rows.append(qd[:, a]); cols.append(qd[:, b_]); vals.append(m * M[a, b_])
        for r in range(pd + 1):
            for a in range(fd + 1):
                rows.append(pdofs[:, r]); cols.append(qd[:, a]); vals.append(np.full(nc, B[r, a]))
                rows.append(qd[:, a]); cols.append(pdofs[:, r]); vals.append(np.full(nc, -B[r, a]))
        u, v = self.edges[:, 0], self.edges[:, 1]
        ein = np.flatnonzero(self.lm_index[v] >= 0)
        eout = np.flatnonzero(self.lm_index[u] >= 0)
        last, first = ein * N + N - 1, eout * N
        for a in range(fd + 1):  # full cell rows incl. explicit zeros (SURVEY A.3)
            lin = self.loff + self.lm_index[v[ein]]
            rows += [lin, qd[last, a]]; cols += [qd[last, a], lin]; vals += [np.full(ein.size, t1[a])] * 2
            lout = self.loff + self.lm_index[u[eout]]
            rows += [lout, qd[first, a]]; cols += [qd[first, a], lout]; vals += [np.full(eout.size, -t0[a])] * 2
        A = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                          shape=(self.n_dofs, self.n_dofs)).tocsr()
        A.sort_indices()
        b = np.zeros(self.n_dofs)
        for r in range(pd + 1):
            np.add.at(b, pdofs[:, r], fc * h * w[r])
        outlet = np.flatnonzero(self.lm_index[v] < 0)
        inlet = np.flatnonzero(self.lm_index[u] < 0)
        np.add.at(b, self.fb[outlet] + N, pbc_vertex[v[outlet]])
        np.add.at(b, self.fb[inlet], -pbc_vertex[u[inlet]])
        return A, b
