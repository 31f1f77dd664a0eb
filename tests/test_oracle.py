"""The CPU oracle pinned against (a) fixtures generated from the reference's own code,
(b) the values the reference's tests assert, (c) closed-form known answers (SURVEY A.6)."""

import pathlib

import networkx as nx
import numpy as np
import pytest

from oracle import reference_port as rp
from tests import helpers

GOLDEN = np.load(pathlib.Path(__file__).parent / "golden" / "reference_graphs.npz")


def golden_graph(key):
    G = nx.DiGraph()
    pos, edges = GOLDEN[key + "/pos"], GOLDEN[key + "/edges"]
    for i, p in enumerate(pos):
        G.add_node(i, pos=p)
    for u, v in edges.tolist():
        G.add_edge(u, v)
    return G


def oracle_net(G, N, strategy=None):
    col = rp.color_graph_literal(G, strategy)
    return rp.OracleNetwork(*rp.graph_to_arrays(G, col), N), col


# ---- (b) the reference's own tests, re-expressed on the oracle -----------------------------------
@pytest.mark.parametrize("N", [10, 50])
def test_edge_info(N):
    """tests/test_edge_info.py:36-55."""
    G = helpers.edge_info_graph()
    col = rp.color_graph_literal(G, None)
    info = rp.analyse_graph_literal(G, col)
    np.testing.assert_array_equal(info.bifurcation_values, [1, 2, 3, 4, 5, 7])
    n_in = np.diff(info.in_offsets)
    n_out = np.diff(info.out_offsets)
    assert list(zip(n_in, n_out)) == [(1, 1), (1, 1), (1, 1), (2, 1), (2, 1), (1, 3)]
    # graph.edges() is adjacency order, not insertion order (SURVEY Appendix C)
    assert list(G.edges()) == [(0, 1), (1, 7), (2, 5), (3, 4), (4, 5), (5, 6), (7, 2), (7, 3), (7, 4)]
    net = rp.OracleNetwork(*rp.graph_to_arrays(G, col), N)
    np.testing.assert_array_equal(net.bifurcation_values, info.bifurcation_values)


@pytest.mark.parametrize("gdim", [2, 3])
@pytest.mark.parametrize("N", [1, 4, 10])
@pytest.mark.parametrize("n", [2, 5, 7])
def test_make_tree_counts(n, gdim, N):
    """tests/test_make_tree.py:14-24: cells = N*(2^n-1), vertices = N+1+(segments-1)*N."""
    G = golden_graph(f"tree_n{n}_H1_W1_d{gdim}")
    net, col = oracle_net(G, N)
    segs = 2**n - 1
    assert net.gdim == gdim
    assert net.cells.shape[0] == N * segs
    assert net.x.shape[0] == N + 1 + (segs - 1) * N
    nodes, cells, markers, orient = rp.mesh_arrays_literal(G, N, col)
    assert np.array_equal(nodes, net.x) and np.array_equal(cells, net.cells)
    assert np.array_equal(markers, net.cell_markers)


@pytest.mark.parametrize("order", ["in", "reverse", "alternating"])
@pytest.mark.parametrize("N", [1, 4, 8])
def test_orientation(order, N):
    """tests/test_orientation.py:27-58: int (1,0).t orientation dx."""
    ordered = {"in": lambda _: True, "reverse": lambda _: False, "alternating": lambda k: k % 2}[order]
    G = helpers.linear_graph(30, ordered=ordered)
    net, _ = oracle_net(G, N)
    val = net.oriented_tangent_integral((1, 0))
    expected = {"in": 1.0, "reverse": -1.0, "alternating": (29 % 2) * -1 / 29}[order]
    assert np.isclose(val, expected)
    assert np.all(net.orientation == 1.0)  # SURVEY A.2: net effect of mesh.py:321-322 and :379-398


# ---- (a) fixtures from the reference's generators --------------------------------------------------
def test_y_mesh_arrays_match_survey():
    """Appendix B: Y-demo mesh arrays restated from mesh.py:270-324."""
    G = golden_graph("tree_n2_H1_W3_d3")
    col = rp.color_graph_literal(G, None)
    nodes, cells, markers, orient = rp.mesh_arrays_literal(G, 4, col)
    np.testing.assert_allclose(nodes[:4], [(0, 0, 0), (0, 0.5, 0), (-1.5, 1, 0), (1.5, 1, 0)])
    assert cells.tolist()[:5] == [[0, 4], [4, 5], [5, 6], [6, 1], [1, 7]] and cells.tolist()[-1] == [12, 3]
    assert markers.tolist() == [0] * 4 + [1] * 4 + [2] * 4
    assert orient.tolist() == [1, 1, 1, -1] * 3  # input signs; the net orientation is +1
    info = rp.analyse_graph_literal(G, col)
    assert info.bifurcation_values.tolist() == [1] and info.boundary_values.tolist() == [0, 2, 3]
    assert info.in_color.tolist() == [0] and info.out_color.tolist() == [1, 2]
    assert info.boundary_in_nodes.tolist() == [2, 3] and info.boundary_out_nodes.tolist() == [0]
    tags, im, om = rp.vertex_markers_literal(info)
    assert (im, om) == (12, 20) and tags.tolist() == [20, 1, 12, 12]
    infl, outfl = rp.integration_entities_literal(G, 4, col, info)
    assert infl[0].tolist() == [3, 1] and outfl[1].tolist() == [4, 0] and outfl[2].tolist() == [8, 0]


@pytest.mark.parametrize("key,N,strategy", [
    ("tree_n3_H1_W1_d2", 1, None), ("tree_n3_H2_W1_d3", 3, "smallest_last"),
    ("tree_n5_H1_W3_d3", 2, "largest_first"), ("arterial_N3_g0.8_d0_1_0", 4, "largest_first"),
])
def test_vectorised_assembly_equals_literal(key, N, strategy):
    G = golden_graph(key)
    net, col = oracle_net(G, N, strategy)
    p = lambda x: x[1] + 0.25 * x[0]  # noqa: E731
    A, b = net.assemble(net.eval_pbc(p), R=1.7, f=0.3)
    Ad, bd, stored = rp.assemble_literal(G, N, col, p, R=1.7, f=0.3)
    assert np.array_equal(A.toarray(), Ad) and np.array_equal(b, bd)
    P = np.zeros_like(stored)
    coo = A.tocoo()
    P[coo.row, coo.col] = True
    assert np.array_equal(P, stored), "pattern (incl. explicit zeros) differs"
    assert A.nnz == net.expected_nnz()
    assert A.has_sorted_indices


def test_sizes_match_survey_appendix_b():
    for key, N, dofs, nnz in [("tree_n2_H1_W3_d3", 4, 28, 99), ("tree_n2_H3.1_W7.3_d3", 5, 34, 120),
                              ("tree_n10_H1_W1_d3", 16, 34270, 121731), ("arterial_N5_g0.8_d0.1_1_0", 40, 2526, 8891)]:
        net, _ = oracle_net(golden_graph(key), N)
        assert (net.n_dofs, net.expected_nnz()) == (dofs, nnz)


def test_reference_coloring_fixture():
    """networkx greedy colouring of the line graph (mesh.py:38-39) recorded from the reference call
    sequence: the colouring is proper and uses 3 (sometimes 4) colours on binary trees."""
    for n in (3, 5, 7):
        G = golden_graph(f"tree_n{n}_H1_W1_d3")
        for strat in ("smallest_last", "largest_first"):
            col = GOLDEN[f"color_tree_n{n}_{strat}"]
            mine = rp.color_graph_literal(G, strat)
            assert [rp.lookup_color(mine, u, v) for u, v in G.edges()] == col.tolist()
            assert 3 <= len(set(col.tolist())) <= 4  # max degree 3; greedy may need one more
            for node in G.nodes():
                inc = [c for (u, v), c in zip(G.edges(), col) if node in (u, v)]
                assert len(inc) == len(set(inc))


# ---- (c) known answers -----------------------------------------------------------------------------
def test_kat_y_bifurcation():
    """SURVEY A.6: make_tree(2,1,3), N=4, p_bc = y."""
    net, _ = oracle_net(golden_graph("tree_n2_H1_W3_d3"), 4)
    A, b = net.assemble(net.eval_pbc(lambda x: x[1]))
    q0, q1, q2, p, lam = net.split(net.solve(A, b))
    np.testing.assert_allclose(q0, 0.7748517734455862, rtol=1e-13)
    np.testing.assert_allclose(q1, 0.3874258867227931, rtol=1e-13)
    np.testing.assert_allclose(q2, 0.3874258867227931, rtol=1e-13)
    np.testing.assert_allclose(lam, [-0.3874258867227931], rtol=1e-13)
    np.testing.assert_allclose(p[:4], [-0.04842824, -0.14528471, -0.24214118, -0.33899765], atol=1e-8)


def test_kat_double_y():
    """make_tree(2,3.1,7.3), N=5, p_bc = x: q = (0, -0.920444352, +0.920444352), lambda = 0."""
    net, _ = oracle_net(golden_graph("tree_n2_H3.1_W7.3_d3"), 5)
    A, b = net.assemble(net.eval_pbc(lambda x: x[0]))
    q0, q1, q2, p, lam = net.split(net.solve(A, b))
    np.testing.assert_allclose(q0, 0.0, atol=1e-14)
    np.testing.assert_allclose(q1, -0.920444352, atol=1e-9)
    np.testing.assert_allclose(q2, 0.920444352, atol=1e-9)
    np.testing.assert_allclose(lam, 0.0, atol=1e-14)


@pytest.mark.parametrize("seed", [0, 1])
def test_resistor_network_closed_form(seed):
    """f = 0: the discrete solution is the resistor network with boundary pressures -p_bc; q is
    constant per edge, Kirchhoff holds at every bifurcation, p follows p_{j+1} = p_j - R q h."""
    G = helpers.random_tree(60, seed)
    net, _ = oracle_net(G, 3, "smallest_last")
    rng = np.random.default_rng(seed)
    R = rng.uniform(0.5, 2.0, net.cells.shape[0])
    pbc = net.eval_pbc(lambda x: x[0] - x[2])
    A, b = net.assemble(pbc, R=R)
    x = net.solve(A, b)
    q_edge, lam = net.resistor_network_solution(pbc, R=R)
    np.testing.assert_allclose(x[net.loff:], lam, rtol=1e-10, atol=1e-13)
    for a in range(4):
        np.testing.assert_allclose(x[net.fb + a], q_edge, rtol=1e-9, atol=1e-12)
    assert np.linalg.norm(A @ x - b) <= 1e-12 * np.linalg.norm(b)
    lam_rows = A[net.loff:]
    assert np.abs(lam_rows @ x).max() < 1e-12  # flux conservation at every bifurcation
    h = net.cell_lengths().reshape(net.E, 3)
    p = x[net.poff:net.loff].reshape(net.E, 3)
    np.testing.assert_allclose(p[:, 1] - p[:, 0], -(R.reshape(net.E, 3)[:, :2] * h[:, :2]).sum(1) / 2 * q_edge, rtol=1e-8, atol=1e-11)


def test_symmetrised_system():
    """SURVEY A.1: negating the pressure rows gives a symmetric matrix with the same solution."""
    net, _ = oracle_net(golden_graph("tree_n5_H1_W1_d3"), 2, "smallest_last")
    A, b = net.assemble(net.eval_pbc(lambda x: x[1]))
    S = A.tolil()
    S[net.poff:net.loff] = -S[net.poff:net.loff]
    S = S.tocsr()
    assert abs(S - S.T).max() < 1e-15
    assert abs(A - A.T).max() == 2.0


# ---- second derivation of the element tensors: FFCx-style quadrature from the coordinate dofs ---------
@pytest.mark.parametrize("fd,pd", [(1, 0), (2, 1), (2, 0), (3, 2), (4, 3)])
def test_closed_form_element_tensors_equal_the_quadrature_literal(fd, pd):
    """R h M_ref / B_ref / f h w_ref (what reference_port.py, elements.py and the CUDA kernels use) against
    Gauss quadrature with detJ = ||J||, K = J^T/||J||^2 on randomly placed cells in 3-D; B does not depend
    on the cell; the orientation flips B only."""
    from networks_fenicsx_b200 import elements
    from oracle import ffcx_literal

    rng = np.random.default_rng(10 * fd + pd)
    M_ref, B_ref, w_ref, _, _ = rp.lagrange_tables(fd, pd)
    M_prod, B_prod, w_prod, _, _ = elements.tables(fd, pd)
    for _ in range(5):
        x0, x1 = rng.normal(size=3), rng.normal(size=3)
        R, f = float(rng.uniform(0.1, 5.0)), float(rng.normal())
        h = np.linalg.norm(x1 - x0)
        M, B, L = ffcx_literal.cell_tensors(x0, x1, fd, pd, R=R, f=f)
        for Mt, Bt, wt in ((M_ref, B_ref, w_ref), (M_prod, B_prod, w_prod)):
            np.testing.assert_allclose(M, R * h * Mt, rtol=1e-12, atol=1e-14)
            np.testing.assert_allclose(B, Bt, rtol=1e-12, atol=1e-13)
            np.testing.assert_allclose(L, f * h * wt, rtol=1e-12, atol=1e-14)
        Mf, Bf, _ = ffcx_literal.cell_tensors(x0, x1, fd, pd, R=R, f=f, orientation=-1.0)
        np.testing.assert_allclose(Bf, -B, rtol=0, atol=1e-15)
        np.testing.assert_allclose(Mf, M, rtol=0, atol=0)
    if (fd, pd) == (1, 0):
        np.testing.assert_allclose(M_ref, [[1 / 3, 1 / 6], [1 / 6, 1 / 3]], rtol=1e-15)
        np.testing.assert_allclose(B_ref, [[-1.0, 1.0]], rtol=1e-15)


@pytest.mark.parametrize("fd,pd", [(1, 0), (2, 1), (3, 2), (2, 0)])
def test_vectorised_assembly_equals_the_cellwise_quadrature_assembly(fd, pd):
    """The COO assembly of the oracle (reference tables x R h, vectorised over cells) against a DOLFINx-style
    cell loop with quadrature-tabulated element tensors and dense accumulation: values of A (explicit zeros
    aside) and b agree to rounding on a Y bifurcation, a random tree and the cyclic test graph."""
    from oracle import ffcx_literal

    rng = np.random.default_rng(3 * fd + pd)
    from networks_fenicsx_b200 import network_generation as ng

    for G, N, strategy in ((ng.make_tree(2, 1, 3), 3, None), (helpers.random_tree(25, 5), 2, "smallest_last"),
                           (helpers.edge_info_graph(), 2, "largest_first")):
        coloring = rp.color_graph_literal(G, strategy)
        pos, edges, colors = rp.graph_to_arrays(G, coloring)
        net = rp.OracleNetworkHO(pos, edges, colors, N, fd, pd) if (fd, pd) != (1, 0) else rp.OracleNetwork(pos, edges, colors, N)
        nc = N * edges.shape[0]
        R, f = rng.uniform(0.5, 2.0, nc), rng.normal(size=nc)
        pbc = net.eval_pbc(lambda x: x[1] - 0.3 * x[0])
        A, b = net.assemble(pbc, R=R, f=f)
        Ad, bd = ffcx_literal.assemble_cellwise(net, pbc, R=R, f=f)
        np.testing.assert_allclose(A.toarray(), Ad, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(b, bd, rtol=1e-12, atol=1e-13)


# ---- the high-precision references the GPU operator tests compare against ---------------------------------------
def _fraction_solve(A, b):
    """Exact solution of A x = b by Gaussian elimination over the rationals (A, b: float64 entries, taken exactly)."""
    from fractions import Fraction

    n = A.shape[0]
    M = [[Fraction(float(v)) for v in row] + [Fraction(float(bi))] for row, bi in zip(A.toarray(), b)]
    for c in range(n):
        p = next(i for i in range(c, n) if M[i][c] != 0)
        M[c], M[p] = M[p], M[c]
        piv = M[c]
        for i in range(c + 1, n):
            if M[i][c] != 0:
                f = M[i][c] / piv[c]
                M[i] = [a - f * bb for a, bb in zip(M[i], piv)] if f else M[i]
    x = [Fraction(0)] * n
    for i in range(n - 1, -1, -1):
        x[i] = (M[i][n] - sum(M[i][j] * x[j] for j in range(i + 1, n))) / M[i][i]
    return x


def _block_errors(net, x, x_exact):
    """Per block (flux, pressure, multipliers): ||x - x_exact|| / ||x_exact||, with x_exact rational and the
    difference formed exactly."""
    from fractions import Fraction

    out = []
    for lo, hi in ((0, net.poff), (net.poff, net.loff), (net.loff, net.n_dofs)):
        d = [Fraction(*np.longdouble(x[i]).as_integer_ratio()) - x_exact[i] for i in range(lo, hi)]
        num = float(sum(v * v for v in d))
        den = float(sum(x_exact[i] * x_exact[i] for i in range(lo, hi)))
        out.append(np.sqrt(num / den))
    return np.asarray(out)


@pytest.mark.parametrize("graph", ["Y", "double_Y"])
@pytest.mark.parametrize("N", [1, 3])
def test_solve_exact_against_rational_elimination(graph, N):
    """solve_exact (float64 SuperLU + refinement with an extended-precision residual) agrees with exact rational
    Gaussian elimination to far below float64 rounding, block by block, on the Y and double-Y systems with a source:
    it is a reference the float64 solvers can be measured against."""
    G = golden_graph("tree_n2_H1_W3_d3") if graph == "Y" else helpers.double_junction_graph()
    net, _ = oracle_net(G, N, "smallest_last")
    rng = np.random.default_rng(7 * N + len(graph))
    nc = net.cells.shape[0]
    A, b = net.assemble(net.eval_pbc(lambda x: x[1] - 0.4 * x[0]), R=rng.uniform(0.5, 2.0, nc), f=rng.normal(size=nc))
    assert np.count_nonzero(b[net.poff:net.loff]) == nc  # f != 0: every pressure row is populated
    x_exact = _fraction_solve(A, b)
    err = _block_errors(net, rp.OracleNetwork.solve_exact(A, b), x_exact)
    err64 = _block_errors(net, net.solve(A, b), x_exact)
    assert err.max() <= 1e-17, err
    assert err64.max() <= 1e-13, err64


def _krylov_min_residual(A, b, dinv, k):
    """min over y in K_k(A D, b) of ||b - A D y||, by a dense float64 least-squares solve on an explicit (column-
    normalised) Krylov basis: an independent statement of what GMRES minimises."""
    cols = [b / np.linalg.norm(b)]
    for _ in range(k - 1):
        v = A @ (dinv * cols[-1])
        cols.append(v / np.linalg.norm(v))
    AK = np.column_stack([A @ (dinv * c) for c in cols])
    y = np.linalg.lstsq(AK, b, rcond=None)[0]
    return np.linalg.norm(b - AK @ y)


@pytest.mark.parametrize("pc", ["none", "jacobi"])
def test_gmres_reference(pc):
    """gmres_reference: the minimal residuals never increase (also across restarts), reach zero at k = n on a small
    system, agree with a least-squares minimisation over an explicit Krylov basis for small k, and the returned
    iterate has the residual it reports."""
    G = golden_graph("tree_n2_H1_W3_d3")
    net, _ = oracle_net(G, 2)
    rng = np.random.default_rng(3)
    nc = net.cells.shape[0]
    A, b = net.assemble(net.eval_pbc(lambda x: x[1]), R=rng.uniform(0.5, 2.0, nc), f=rng.normal(size=nc))
    n = net.n_dofs
    dinv = np.ones(n)
    if pc == "jacobi":
        dinv[:net.poff] = 1.0 / A.diagonal()[:net.poff]
    minv = None if pc == "none" else dinv
    nb = np.linalg.norm(b)
    rho, beta, x = rp.OracleNetwork.gmres_reference(A, b, minv, n, n)
    assert rho.size == n + 1 and beta.size == 2
    assert np.all(np.diff(rho.astype(np.float64)) <= 1e-15 * nb)
    assert rho[-1] <= 1e-14 * nb and beta[-1] <= 1e-14 * nb
    for k in range(1, 6):
        np.testing.assert_allclose(float(rho[k]), _krylov_min_residual(A, b, dinv, k), rtol=1e-8)
    # restarted: the iterate of each cycle is the start of the next, the residuals keep decreasing
    m, k_max = 3, 12
    rho_r, beta_r, x_r = rp.OracleNetwork.gmres_reference(A, b, minv, m, k_max)
    assert rho_r.size == k_max + 1 and beta_r.size == k_max // m + 1
    assert np.all(np.diff(rho_r.astype(np.float64)) <= 1e-15 * nb)
    np.testing.assert_allclose(rho_r[:m + 1].astype(np.float64), rho[:m + 1].astype(np.float64), rtol=1e-12)
    np.testing.assert_allclose(beta_r.astype(np.float64), rho_r[::m].astype(np.float64), rtol=1e-12)
    res = b.astype(np.longdouble) - A.astype(np.longdouble) @ x_r
    np.testing.assert_allclose(float(np.sqrt(np.sum(res * res))), float(rho_r[-1]), rtol=1e-12)
    assert float(rho_r[-1]) > float(rho[k_max])  # restarting costs: GMRES(3) is slower than full GMRES
