"""Higher-order elements on a network cut over several ranks, CPU only:

1. the per-rank table-driven systems sum to the whole network's system (including the nodal pressure rows of
   the shared bifurcations, which are partial sums on every rank);
2. a NumPy emulation of the split top-chunk elimination of condense.cuh (btree_top_split_kernel): per rank the
   kPartial payload, the payloads summed in rank order, kFinish on every rank, back-substitution -- the gathered
   solution is the whole network's direct solve and the replicated nodal unknowns agree bit for bit."""

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200 import condense
from networks_fenicsx_b200 import network_generation as ng
from networks_fenicsx_b200.distributed import partition_tree
from networks_fenicsx_b200.mesh import SerialComm, _greedy_edge_coloring_arrays
from tests import helpers
from tests.ho_partition import expected_exchange_sizes, local_to_global, oracle_ho

DEGREES = [(2, 1), (2, 0), (3, 2)]
P_BC = lambda x: x[1] - 0.5 * x[0]  # noqa: E731


def graph_of(case):
    if case == "tree8":
        return ng.make_tree(8, 3, 5, as_arrays=True)
    if case == "arterial":
        return ng.make_arterial_tree(6, as_arrays=True)
    H = helpers.random_tree(300, 7)
    return ng.ArrayGraph(np.asarray([H.nodes[i]["pos"] for i in H.nodes()]), np.asarray(list(H.edges()), dtype=np.int64))


CASES = [("tree8", 2, 2), ("tree8", 4, 2), ("random", 3, 2), ("arterial", 2, 2), ("arterial", 2, 3)]


def coefficients(G, N):
    E = G.number_of_edges()
    R = 1.0 + 0.5 * np.cos(np.arange(E * N, dtype=np.float64))
    f = 0.3 + np.sin(np.arange(E * N, dtype=np.float64))
    return R, f


@pytest.mark.parametrize("fd,pd", DEGREES)
@pytest.mark.parametrize("case,world,N", CASES)
def test_partitioned_higher_order_assembly_sums_to_global(case, world, N, fd, pd):
    G = graph_of(case)
    R, f = coefficients(G, N)
    gnet = oracle_ho(G.pos, G.edges, _greedy_edge_coloring_arrays(G.number_of_nodes(), G.edges), N, fd, pd)
    A, b = gnet.assemble(gnet.eval_pbc(P_BC), R=R, f=f)
    S = sp.csr_matrix(A.shape)
    bsum = np.zeros_like(b)
    shared_rows = {}
    for rank in range(world):
        part = partition_tree(G, world, rank, chunk_nodes=8)
        colors = _greedy_edge_coloring_arrays(part.graph.number_of_nodes(), part.graph.edges)
        lnet = oracle_ho(part.graph.pos, part.graph.edges, colors, N, fd, pd, degree=part.node_degree)
        cells = (part.global_edges[:, None] * N + np.arange(N)[None, :]).ravel()
        Al, bl = lnet.assemble(lnet.eval_pbc(P_BC), R=R[cells], f=f[cells])
        idx = local_to_global(part, lnet, gnet)
        P = sp.csr_matrix((np.ones(idx.size), (np.arange(idx.size), idx)), shape=(idx.size, gnet.n_dofs))
        S = S + P.T @ Al @ P
        bsum += P.T @ bl
        if pd >= 1:
            nodes = lnet.bifurcation_values[part.shared_lm]
            shared_rows[rank] = dict(zip(part.global_nodes[nodes].tolist(), bl[lnet.poff + nodes]))
    assert abs(S - A).max() < 1e-13
    np.testing.assert_allclose(bsum, b, rtol=0, atol=1e-13)
    if pd >= 1:  # the hazard of the shared right-hand-side rows is exercised: the ranks hold different parts
        differ = [n for n in shared_rows[0] if any(abs(shared_rows[r][n] - shared_rows[0][n]) > 1e-12 for r in range(1, world))]
        assert differ


def rank_state(G, world, rank, N, fd, pd, R, f):
    part = partition_tree(G, world, rank, chunk_nodes=8)
    nm = nxfx.NetworkMesh(part.graph, N=N, color_strategy="smallest_last", node_degree=part.node_degree,
                          comm=SerialComm(), device=0)
    net = oracle_ho(nm._node_pos, nm.graph_edges, nm.edge_colors, N, fd, pd, degree=part.node_degree)
    cells = (part.global_edges[:, None] * N + np.arange(N)[None, :]).ravel()
    _, b = net.assemble(net.eval_pbc(P_BC), R=R[cells], f=f[cells])
    return part, nm, net, condense.build_condensation(nm, fd, pd), R[cells] * net.cell_lengths(), b


def edge_stage(nm, cond, cell_rh, r):
    """Per edge: Y_e, y0_e, S_e, h_e and the global rows of the local unknowns (condense.cuh)."""
    edges, N = nm.graph_edges, cond.N
    per_edge = cond.fd * N + 1
    nq = edges.shape[0] * per_edge
    lm = nm.node_multiplier_index
    out = []
    for e, (u, v) in enumerate(edges):
        t = cond.types[int(lm[u] >= 0) + 2 * int(lm[v] >= 0)]
        K = np.zeros((t.n, t.n))
        np.add.at(K, (t.k_row, t.k_col), t.k_coef * np.where(t.k_cell >= 0, cell_rh[e * N + np.maximum(t.k_cell, 0)], 1.0))
        Cm = np.zeros((t.n, 4))
        np.add.at(Cm, (t.c_row, t.c_slot), t.c_coef)
        Dm = np.zeros((4, t.n))
        np.add.at(Dm, (t.d_slot, t.d_col), t.d_coef)
        g = []
        for kind, off in zip(t.loc_kind, t.loc_off):
            if kind == condense.K_FLUX:
                g.append(nm.edge_slot[e] * per_edge + off)
            elif kind == condense.K_PCELL:
                g.append(cond.pcell_base + e * cond.pcell_stride + off)
            elif kind == condense.K_PVERT:
                g.append(nq + nm._n_nodes + e * (N - 1) + off)
            else:
                g.append(nq + (u if kind == condense.K_PU else v))
        g = np.asarray(g)
        Ye, ye = np.linalg.solve(K, Cm), np.linalg.solve(K, r[g])
        out.append((Ye, ye, -Dm @ Ye, Dm @ ye, g))
    return out, nq


class RankEmulation:
    """One rank of the host-driven partitioned solve: setup + first application (r = b as assembled)."""

    def __init__(self, part, nm, cond, cell_rh, r):
        self.part, self.nm, self.cond = part, nm, cond
        s = self.s = part.schedule
        edges = nm.graph_edges
        lm = nm.node_multiplier_index
        n_bif = nm.bifurcation_values.size
        self.loff = r.size - n_bif
        self.edge, self.nq = edge_stage(nm, cond, cell_rh, r)
        tob = s.t_of_bif
        self.D0 = np.zeros((n_bif, 2, 2))
        self.rz = np.zeros((n_bif, 2))
        for b in range(n_bif):  # P rows unweighted (additive), multiplier rows weighted by ownership
            self.rz[tob[b]] = [r[self.nq + nm.bifurcation_values[b]] if cond.pd >= 1 else 0.0,
                               part.lam_weight[b] * r[self.loff + b]]
        for e, (u, v) in enumerate(edges):
            S, h = self.edge[e][2], self.edge[e][3]
            if lm[u] >= 0:
                self.D0[tob[lm[u]]] += S[0:2, 0:2]
                self.rz[tob[lm[u]]] -= h[0:2]
            if lm[v] >= 0:
                self.D0[tob[lm[v]]] += S[2:4, 2:4]
                self.rz[tob[lm[v]]] -= h[2:4]
        if cond.pd == 0:
            self.D0[:, 0, 0] = 1.0
        self.U = np.zeros((n_bif, 2, 2))
        self.L = np.zeros((n_bif, 2, 2))
        bif_of_t = np.argsort(tob)
        for t_ in range(n_bif):
            pe = s.t_pedge[t_]
            if pe < 0:
                continue
            Se = self.edge[pe][2]
            if lm[edges[pe][0]] == bif_of_t[t_]:
                self.U[t_], self.L[t_] = Se[0:2, 2:4], Se[2:4, 0:2]
            else:
                self.U[t_], self.L[t_] = Se[2:4, 0:2], Se[0:2, 2:4]
        self.Dinv, self.G, self.H = (np.zeros((n_bif, 2, 2)) for _ in range(3))
        self.z = np.zeros((n_bif, 2))
        top = s.n_chunks - 1
        self.b0 = s.lvl_ptr[s.chunk_lptr[top]]
        self.sh_idx = np.full(n_bif - self.b0, -1)
        self.sh_idx[tob[part.shared_lm] - self.b0] = np.arange(part.shared_lm.size)
        self.nt = max(part.shared_lm.size, 1)

    def k(self, n):
        return -1 if n < self.b0 else int(self.sh_idx[n - self.b0])

    def levels(self, c):
        return range(self.s.chunk_lptr[c], self.s.chunk_lptr[c + 1])

    def nodes(self, lv):
        return range(self.s.lvl_ptr[lv], self.s.lvl_ptr[lv + 1])

    def children(self, n):
        return self.s.t_cidx[self.s.t_cptr[n]:self.s.t_cptr[n + 1]]

    def eliminate(self, n, Dn):
        self.Dinv[n] = np.linalg.inv(Dn)
        self.G[n] = self.Dinv[n] @ self.U[n]
        self.H[n] = self.L[n] @ self.Dinv[n]

    def partial(self):
        """Bottom chunks, then kPartial of the top chunk; returns [D | U | L | rhs] (setup + apply sections)."""
        s, nt = self.s, self.nt
        for c in range(s.n_chunks - 1):
            for lv in reversed(self.levels(c)):
                for n in self.nodes(lv):
                    Dn = self.D0[n].copy()
                    for ch in self.children(n):
                        Dn -= self.H[ch] @ self.U[ch]
                        self.rz[n] -= self.H[ch] @ self.rz[ch]
                    self.eliminate(n, Dn)
        buf = np.zeros(14 * nt)
        for lv in reversed(self.levels(s.n_chunks - 1)):
            for n in self.nodes(lv):
                Dn = self.D0[n].copy()
                for ch in self.children(n):
                    if self.k(ch) < 0:
                        Dn -= self.H[ch] @ self.U[ch]
                        self.rz[n] -= self.H[ch] @ self.rz[ch]
                k = self.k(n)
                if k < 0:
                    self.eliminate(n, Dn)
                else:
                    buf[4 * k:4 * k + 4] = Dn.ravel()
                    buf[4 * nt + 4 * k:4 * nt + 4 * k + 4] = self.U[n].ravel()
                    buf[8 * nt + 4 * k:8 * nt + 4 * k + 4] = self.L[n].ravel()
                    buf[12 * nt + 2 * k:12 * nt + 2 * k + 2] = self.rz[n]
        return buf

    def finish(self, buf):
        """kFinish of the top chunk from the summed payload, the backward sweeps, the back-substitution."""
        s, nt = self.s, self.nt
        top = s.n_chunks - 1
        for lv in reversed(self.levels(top)):
            for n in self.nodes(lv):
                k = self.k(n)
                if k < 0:
                    continue
                Dn = buf[4 * k:4 * k + 4].reshape(2, 2).copy()
                r = buf[12 * nt + 2 * k:12 * nt + 2 * k + 2].copy()
                shared = sorted((self.k(ch), ch) for ch in self.children(n) if self.k(ch) >= 0)
                for _, ch in shared:  # exchanged order: the same operations on every rank
                    Dn -= self.H[ch] @ self.U[ch]
                    r -= self.H[ch] @ self.rz[ch]
                if self.cond.pd == 0:
                    Dn[0, 0], Dn[0, 1], Dn[1, 0] = 1.0, 0.0, 0.0
                self.U[n] = buf[4 * nt + 4 * k:4 * nt + 4 * k + 4].reshape(2, 2)
                self.L[n] = buf[8 * nt + 4 * k:8 * nt + 4 * k + 4].reshape(2, 2)
                self.eliminate(n, Dn)
                self.rz[n] = r
        for c in [top, *range(top)]:
            for lv in self.levels(c):
                for n in self.nodes(lv):
                    self.z[n] = self.Dinv[n] @ self.rz[n]
                    if s.t_parent[n] >= 0:
                        self.z[n] -= self.G[n] @ self.z[s.t_parent[n]]
        nm, tob = self.nm, s.t_of_bif
        lm = nm.node_multiplier_index
        x = np.zeros(self.loff + nm.bifurcation_values.size)
        for e, (u, v) in enumerate(nm.graph_edges):
            ze = np.zeros(4)
            if lm[u] >= 0:
                ze[0:2] = self.z[tob[lm[u]]]
            if lm[v] >= 0:
                ze[2:4] = self.z[tob[lm[v]]]
            Ye, ye, _, _, g = self.edge[e]
            x[g] = ye - Ye @ ze
        for b in range(nm.bifurcation_values.size):
            if self.cond.pd >= 1:
                x[self.nq + nm.bifurcation_values[b]] = self.z[tob[b], 0]
            x[self.loff + b] = self.z[tob[b], 1]
        return x


@pytest.mark.parametrize("fd,pd", DEGREES)
@pytest.mark.parametrize("case,world,N", CASES)
def test_partitioned_condensation_emulation_is_the_global_direct_solve(case, world, N, fd, pd):
    G = graph_of(case)
    R, f = coefficients(G, N)
    gnet = oracle_ho(G.pos, G.edges, _greedy_edge_coloring_arrays(G.number_of_nodes(), G.edges), N, fd, pd)
    A, b = gnet.assemble(gnet.eval_pbc(P_BC), R=R, f=f)
    x_ref = spla.spsolve(A.tocsc(), b)
    ranks, payloads = [], []
    for rank in range(world):
        part, nm, net, cond, cell_rh, bl = rank_state(G, world, rank, N, fd, pd, R, f)
        emu = RankEmulation(part, nm, cond, cell_rh, bl)
        payloads.append(emu.partial())
        setup, apply, _ = expected_exchange_sizes(part.n_top, pd >= 1)
        assert payloads[-1].size == setup + apply
        ranks.append((part, net, emu))
    total = payloads[0].copy()
    for p in payloads[1:]:  # the all-reduce, in rank order
        total += p
    x = np.full(gnet.n_dofs, np.nan)
    replicated = []
    for part, net, emu in ranks:
        xl = emu.finish(total.copy())
        idx = local_to_global(part, net, gnet)
        x[idx] = xl
        sh = part.shared_lm
        replicated.append(np.concatenate([emu.z[part.schedule.t_of_bif[sh]].ravel(), xl[emu.loff + sh]]))
    assert not np.isnan(x).any()
    for rep in replicated[1:]:
        assert np.array_equal(rep, replicated[0]), "the replicated nodal unknowns differ between ranks"
    assert helpers.rel_l2(x, x_ref) < 1e-10, helpers.rel_l2(x, x_ref)
