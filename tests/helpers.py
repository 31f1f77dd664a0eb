"""Shared graph builders / comparison helpers for the tests."""

import socket

import networkx as nx
import numpy as np

from oracle import reference_port as rp


def edge_info_graph():
    """The 8-node cyclic graph of the reference's tests/test_edge_info.py:12-33."""
    G = nx.DiGraph()
    G.add_node(0, pos=np.zeros(3))
    G.add_node(1, pos=np.array([0.0, 0.0, 1.0]))
    G.add_node(2, pos=np.array([0.2, 0.2, 2.0]))
    G.add_node(3, pos=np.array([-0.2, 0.3, 2.0]))
    G.add_node(4, pos=np.array([0.0, 0.1, 2.1]))
    G.add_node(5, pos=np.array([0.1, -0.1, 3.0]))
    G.add_node(6, pos=np.array([-0.3, 0.4, 4.0]))
    G.add_node(7, pos=1.1 * G.nodes[1]["pos"])
    for e in [(0, 1), (1, 7), (7, 2), (2, 5), (7, 3), (3, 4), (4, 5), (7, 4), (5, 6)]:
        G.add_edge(*e)
    return G


def linear_graph(n: int, dim: int = 2, ordered=lambda _: True) -> nx.DiGraph:
    """tests/test_orientation.py:10-25 of the reference."""
    G = nx.DiGraph()
    G.add_nodes_from(range(n))
    for i in range(n - 1):
        if ordered(i):
            G.add_edge(i, i + 1)
        else:
            G.add_edge(i + 1, i)
    for i in range(n):
        pos = np.zeros(dim)
        pos[0] = i / (n - 1)
        G.nodes[i]["pos"] = pos
    return G


def double_junction_graph():
    """Two junctions: 0->1, 1->2, 1->3, 3->4, 3->5 (SURVEY 8d note on the 'double Y' config)."""
    G = nx.DiGraph()
    pts = [(0, 0, 0), (0, 1, 0), (-1, 2, 0), (1, 2, 0), (0.5, 3, 0.2), (1.7, 3.1, -0.1)]
    for i, p in enumerate(pts):
        G.add_node(i, pos=np.array(p, dtype=float))
    for e in [(0, 1), (1, 2), (1, 3), (3, 4), (3, 5)]:
        G.add_edge(*e)
    return G


def random_tree(n_nodes: int, seed: int, dim: int = 3):
    """Random recursive tree with node 0 as single inlet of degree 1, random edge directions off."""
    rng = np.random.default_rng(seed)
    G = nx.DiGraph()
    for i in range(n_nodes):
        G.add_node(i, pos=rng.normal(size=dim))
    G.add_edge(0, 1)
    for k in range(2, n_nodes):
        G.add_edge(int(rng.integers(1, k)), k)
    return G


def oracle_for(nm, N, G=None, strategy=None):
    """OracleNetwork for the network ``nm`` was built from.

    With the original graph ``G`` the oracle does its OWN graph analysis (node / edge order, colouring
    call of mesh.py:29-42 through ``color_graph_literal``), so that edge ordering or colouring bugs of
    the product cannot cancel out; it then only checks that both agree.  Without ``G`` (or for graphs
    beyond the size networkx colours in reasonable time) it falls back to the product's arrays."""
    from networks_fenicsx_b200.network_generation import ArrayGraph

    if G is None:
        return rp.OracleNetwork(nm._node_pos, nm.graph_edges, nm.edge_colors, N)
    graph = G.to_networkx() if isinstance(G, ArrayGraph) else G
    if graph.number_of_edges() > 20000:
        return rp.OracleNetwork(nm._node_pos, nm.graph_edges, nm.edge_colors, N)
    coloring = rp.color_graph_literal(graph, strategy)
    if isinstance(G, ArrayGraph):  # the arrays ARE the input: their order stands, only the colouring is redone
        pos, edges = np.asarray(G.pos, dtype=np.float64), np.asarray(G.edges, dtype=np.int64)
        if strategy is None:
            colors = np.arange(edges.shape[0], dtype=np.int32)
        else:
            colors = np.asarray([rp.lookup_color(coloring, int(u), int(v)) for u, v in edges], dtype=np.int32)
    else:
        pos, edges, colors = rp.graph_to_arrays(graph, coloring)
    assert np.array_equal(edges, nm.graph_edges), "edge order differs from graph.edges()"
    assert np.array_equal(colors, nm.edge_colors), "edge colouring differs from the reference's call"
    assert np.array_equal(pos, nm._node_pos)
    return rp.OracleNetwork(pos, edges, colors, N)


def free_port() -> int:
    """A loopback TCP port that is free now, for the rendezvous of multi-process tests (a fixed port
    collides with another run of the suite on the same host)."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def rel_l2(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))
