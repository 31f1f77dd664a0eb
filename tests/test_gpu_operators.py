"""The solver's operators against a high-precision reference, on inputs no assembled system produces.

The parity tests solve assembled systems, whose right-hand sides are zero in most rows (multipliers, interior flux
rows, pressure rows when f = 0); the solve repairs small preconditioner errors by refinement or extra FGMRES
iterations.  Here each operator is compared with an exact statement of what it computes:

* the network-Schur preconditioner z = P^{-1} r, an exact solve on trees, for r with one block populated at a time,
  through the stored factors (``nxfx_pc_setup`` + ``nxfx_pc_apply``) and through the factor-and-solve of a fresh
  matrix (``nxfx_solve`` preonly without refinement), on every dispatch branch -- each case asserts the launch
  counts that identify its branch, so a later dispatch change cannot silently drop the coverage;
* FGMRES's residual history against GMRES(m) run in extended precision;
* the residual kernel and the two norms the host's refinement decision reads.

The reference always solves the matrix as stored on the device (``getValuesCSR``), which the parity tests pin to
the oracle's assembly.
"""

import ctypes as C
import math

import networkx as nx
import numpy as np
import pytest

import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200 import _lib
from networks_fenicsx_b200 import network_generation as ng
from networks_fenicsx_b200.schedule import build_tree_schedule
from oracle import reference_port as rp
from tests import helpers

pytestmark = pytest.mark.gpu

P_BC = lambda x: x[1] - 0.3 * x[0] + 0.5  # noqa: E731
exact_solve = rp.OracleNetwork.solve_exact
EPS = float(np.finfo(np.float64).eps)


def _graph(points, edges):
    G = nx.DiGraph()
    for i, p in enumerate(points):
        G.add_node(i, pos=np.asarray(p, dtype=float))
    for e in edges:
        G.add_edge(*e)
    return G


def single_edge():
    return _graph([(0, 0, 0), (1, 2, 0.5)], [(0, 1)])


def star(k=6):
    """Inlet -> hub -> k outlets: one bifurcation of degree k + 1."""
    pts = [(0, 0, 0), (0, 1, 0)] + [(np.cos(a), 2 + np.sin(a), 0.1 * a) for a in np.linspace(0, 3, k)]
    return _graph(pts, [(0, 1)] + [(1, 2 + j) for j in range(k)])


def hub_of_ys(k=100):
    """Inlet -> hub -> k children, each a Y bifurcation with two outlets: a degree-(k+1) node above k nodes."""
    rng = np.random.default_rng(k)
    pts = [(0, 0, 0), (0, 1, 0)]
    edges = [(0, 1)]
    for j in range(k):
        c = len(pts)
        pts += [tuple(rng.normal(size=3) + (0, 3, 0)), tuple(rng.normal(size=3) + (0, 5, 0)), tuple(rng.normal(size=3) + (0, 5, 1))]
        edges += [(1, c), (c, c + 1), (c, c + 2)]
    return _graph(pts, edges)


def random_oriented_tree(seed):
    """Random recursive tree with random edge directions: several inlets and outlets."""
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(20, 60))
    G = nx.DiGraph()
    for i in range(n):
        G.add_node(i, pos=rng.normal(size=3))
    for k in range(1, n):
        p = 0 if k == 1 else int(rng.integers(0, k))
        G.add_edge(*((p, k) if rng.random() < 0.5 else (k, p)))
    return G


class System:
    """One network on its own device context: the solver, its matrix as stored on the device, block bounds."""

    def __init__(self, G, N, fd=1, pd=0, R=None, f=None, chunk_nodes=None, extra_R=0, seed=0, strategy="smallest_last"):
        self.nm = nm = nxfx.NetworkMesh(G, N=N, color_strategy=strategy)
        self.asm = asm = nxfx.HydraulicNetworkAssembler(nm, flux_degree=fd, pressure_degree=pd)
        rng = np.random.default_rng(seed)
        nc = N * G.number_of_edges()
        self.R = [rng.uniform(0.5, 2.0, nc) if R is None else R] + [rng.uniform(0.1, 3.0, nc) for _ in range(extra_R)]
        self.f = rng.normal(size=nc) if f is None else f
        sched = None
        if chunk_nodes is not None:
            sched = build_tree_schedule(nm.graph_edges, nm.node_multiplier_index, nm.bifurcation_values.size,
                                        root_hint_nodes=nm._boundary_out_nodes, chunk_nodes=chunk_nodes)
        asm.compute_forms(p_bc_ex=P_BC, R=self.R[0], f=self.f)
        self.solver = nxfx.Solver(asm, schedule=sched, petsc_options={"ksp_type": "preonly", "pc_type": "lu"})
        self.assemble()
        self.dev = nm.device
        self.n = asm.num_dofs
        nq = sum(asm.block_sizes[:-2])
        npr = asm.block_sizes[-2]
        self.blocks = {"flux": (0, nq), "pressure": (nq, nq + npr), "multipliers": (nq + npr, self.n)}
        self.A = self.solver.A.to_scipy()
        self.schedule = self.solver._schedule
        # longest chain of dependent eliminations: tree levels, then the flux dofs along one edge
        self.path = (int(self.schedule.depth.max()) + 1 if self.schedule.depth.size else 0) + N * fd

    def assemble(self):
        """A fresh matrix: one assembly, then the accumulated ones (ADD_VALUES) with the other resistances."""
        asm, solver = self.asm, self.solver
        asm.compute_forms(p_bc_ex=P_BC, R=self.R[0], f=self.f)
        solver.assemble()
        for R in self.R[1:]:
            asm.compute_forms(p_bc_ex=P_BC, R=R, f=self.f)
            asm.assemble(solver.A, solver.b)
        solver.A._materialise_zero()
        solver.A.bind()
        assert solver.A.accumulated == len(self.R)

    def rhs(self, kind, seed):
        """r with only the rows of one block populated (``nodal``: the pressure rows of the graph nodes' vertices,
        continuous pressure only)."""
        rng = np.random.default_rng(seed)
        r = np.zeros(self.n)
        if kind == "all":
            r[:] = rng.normal(size=self.n)
        elif kind == "nodal":
            p0 = self.blocks["pressure"][0]
            nodes = np.arange(self.nm._node_pos.shape[0])
            r[p0 + nodes] = rng.normal(size=nodes.size)
        else:
            lo, hi = self.blocks[kind]
            r[lo:hi] = rng.normal(size=hi - lo)
        return r

    def block_errors(self, z, x_ref):
        out = {}
        for name, (lo, hi) in self.blocks.items():
            if hi > lo:
                d = z[lo:hi].astype(np.longdouble) - x_ref[lo:hi]
                out[name] = float(np.sqrt(np.sum(d * d) / np.sum(x_ref[lo:hi] * x_ref[lo:hi])))
        return out

    # ---- the two entry points of P^{-1} --------------------------------------------------------------------------
    def pc_apply_stored(self, r):
        """nxfx_pc_setup, then z = P^{-1} r with the stored factors; z pre-filled with NaN.  Returns
        (z, setup launches, apply launches)."""
        dev = self.dev
        self.solver.A.bind()
        rd, zd = dev.from_host(r), dev.from_host(np.full(self.n, np.nan))
        l0 = dev.launch_count
        dev.call("nxfx_pc_setup")
        l1 = dev.launch_count
        dev.call("nxfx_pc_apply", rd.c_ptr, zd.c_ptr)
        l2 = dev.launch_count
        z = zd.download()
        assert np.array_equal(rd.download(), r), "nxfx_pc_apply modified r"
        return z, l1 - l0, l2 - l1

    def pc_apply_fresh(self, r):
        """A freshly assembled matrix and nxfx_solve (preonly, no refinement, final residual): x = P^{-1} b for
        b := r, factorised while eliminating b where the dispatch fuses the two.  Returns (x, launches, info)."""
        self.assemble()
        dev = self.dev
        o = self.solver.ksp.options
        o.update({"nxfx_refine_steps": 0, "nxfx_final_residual": True})
        opts = self.solver.solve_options()
        info = _lib.SolveInfo()
        bd, xd = dev.from_host(r), dev.from_host(np.full(self.n, np.nan))
        l0 = dev.launch_count
        dev.call("nxfx_solve", bd.c_ptr, xd.c_ptr, C.byref(opts), C.byref(info))
        launches = dev.launch_count - l0
        x = xd.download()
        assert np.array_equal(bd.download(), r), "nxfx_solve modified b"
        assert info.iterations == 1
        return x, launches, info


def _superlu_errors(s, r, x_ref):
    return s.block_errors(rp.OracleNetwork.solve(s.A, r), x_ref)


# (id, graph builder, N, (fd, pd), chunk_nodes, extra assemblies, launches of (setup, apply, fresh solve))
# fresh solve = the fused factor-and-solve + residual where can_fuse_setup holds, else setup + apply + residual.
# P1/DG0 apply: bif_rhs_n1 (or edge_condense + bif_rhs) + tree pass + back-substitution;
# higher order apply: edge rhs + node rhs [+ bottom sweep] + top sweep [+ bottom sweep] + back-substitution.
CASES = [
    # N = 1, one chunk: bif_rhs_n1 + tree_solve_kernel<Up> + back-substitution
    ("n1_one_chunk", lambda: ng.make_tree(6, 3, 4), 1, (1, 0), None, 0, (1, 3, 5)),
    # N = 1, several resident chunks: rhs fused into tree_solve_coop_kernel; fused tree_factor_solve_coop_kernel
    ("n1_coop_chunks", lambda: ng.make_tree(8, 3, 4), 1, (1, 0), 16, 0, (1, 2, 3)),
    # N = 1, more chunks than resident blocks: tree_solve_kernel<Up> + <Down>; fused kernel, several chunks per block
    ("n1_many_chunks", lambda: ng.make_tree(14, 3, 5, as_arrays=True), 1, (1, 0), 4, 0, (1, 4, 3)),
    # N >= 2: edge_condense + bif_rhs (+ edge_conductance, bif_diag in the setup; their <true> forms when fused)
    ("n2_one_chunk", lambda: ng.make_tree(6, 3, 4), 2, (1, 0), None, 0, (3, 4, 8)),
    ("n2_coop_chunks", lambda: ng.make_tree(8, 3, 4), 2, (1, 0), 16, 0, (3, 4, 5)),
    ("n3_coop_chunks", lambda: ng.make_tree(8, 3, 4), 3, (1, 0), 16, 0, (3, 4, 5)),
    ("n7_coop_chunks", lambda: ng.make_tree(7, 3, 4), 7, (1, 0), 8, 0, (3, 4, 5)),
    # no shared-memory schedule (chunks deeper than kLevelCap = 64 levels):
    # tree_sweep_kernel<kTreeFactor> x 2, <kTreeUp>, <kTreeUpDown>, <kTreeDown>
    ("chain_global_sweeps_n1", lambda: helpers.linear_graph(400, dim=3), 1, (1, 0), 150, 0, (4, 6, 11)),
    ("chain_global_sweeps_n3", lambda: helpers.linear_graph(400, dim=3), 3, (1, 0), 150, 0, (4, 6, 11)),
    # no bifurcation: the edge kernels only
    ("single_edge_n1", single_edge, 1, (1, 0), None, 0, (1, 2, 4)),
    ("single_edge_n5", single_edge, 5, (1, 0), None, 0, (1, 2, 4)),
    # accumulated matrices (2 and 3 assemblies, other R each time): scale_tail_kernel around the application
    ("accumulated2_n1", lambda: ng.make_tree(7, 3, 4), 1, (1, 0), None, 1, (1, 5, 7)),
    ("accumulated3_n1", lambda: ng.make_tree(7, 3, 4), 1, (1, 0), None, 2, (1, 5, 7)),
    ("accumulated3_n3", lambda: ng.make_tree(7, 3, 4), 3, (1, 0), None, 2, (3, 6, 10)),
    ("accumulated2_n2_chunks", lambda: ng.make_tree(8, 3, 4), 2, (1, 0), 16, 1, (3, 6, 10)),
    # shapes
    ("star6_n1", star, 1, (1, 0), None, 0, (1, 3, 5)),
    ("star6_n3", star, 3, (1, 0), None, 0, (3, 4, 8)),
    ("hub_of_100_ys_n2", hub_of_ys, 2, (1, 0), None, 0, (3, 4, 8)),
    ("random_oriented_0_n1", lambda: random_oriented_tree(0), 1, (1, 0), None, 0, (1, 3, 5)),
    ("random_oriented_1_n2", lambda: random_oriented_tree(1), 2, (1, 0), None, 0, (3, 4, 8)),
    ("random_oriented_2_n4", lambda: random_oriented_tree(2), 4, (1, 0), None, 0, (3, 4, 8)),
    # higher order: edge LU + 2 x 2 node blocks over the same schedule
    ("p2p1_random", lambda: helpers.random_tree(60, 3), 2, (2, 1), None, 0, (3, 4, 8)),
    ("p2dg0_random", lambda: helpers.random_tree(60, 4), 2, (2, 0), None, 0, (3, 4, 8)),
    ("p3p2_random", lambda: helpers.random_tree(60, 5), 2, (3, 2), None, 0, (3, 4, 8)),
    ("p2p1_chunks", lambda: ng.make_tree(8, 3, 4), 2, (2, 1), 16, 0, (4, 6, 11)),
    ("p2p1_accumulated2", lambda: helpers.random_tree(50, 11), 3, (2, 1), None, 1, (3, 6, 10)),
    # 40 cells per edge: the edge band does not fit shared memory, global-memory cond_factor_kernel
    ("p2p1_arterial_n40", lambda: ng.make_arterial_tree(N=5, direction=np.array([0.1, 1.0, 0.0])), 40, (2, 1), None, 0, (3, 4, 8)),
    ("p3p2_arterial_n40", lambda: ng.make_arterial_tree(N=5, direction=np.array([0.1, 1.0, 0.0])), 40, (3, 2), None, 0, (3, 4, 8)),
    ("p2p1_single_edge", single_edge, 3, (2, 1), None, 0, (1, 2, 4)),
    ("p2dg0_single_edge", single_edge, 3, (2, 0), None, 0, (1, 2, 4)),
]


def _check_pc(s, kinds, seed0, floor=1e-13):
    """B1 for one system: every r kind through both entry points against solve_exact.  Returns the worst ratio
    error / bar and the launch counts seen."""
    R = np.column_stack([s.rhs(k, seed0 + i) for i, k in enumerate(kinds)])
    X = exact_solve(s.A, R)
    seen = set()
    worst = {}
    for j, kind in enumerate(kinds):
        r, x_ref = R[:, j], X[:, j]
        lu_err = _superlu_errors(s, r, x_ref)
        bar = {b: max(floor, 100.0 * e, 10.0 * EPS * s.path) for b, e in lu_err.items()}
        z, n_setup, n_apply = s.pc_apply_stored(r)
        x, n_solve, info = s.pc_apply_fresh(r)
        seen.add((n_setup, n_apply, n_solve))
        for entry, v in (("stored factors", z), ("factor-and-solve", x)):
            assert np.isfinite(v).all(), f"{entry}, r = {kind}: entries left unwritten"
            err = s.block_errors(v, x_ref)
            for b, e in err.items():
                assert e <= bar[b], f"{entry}, r = {kind}: {b} block off by {e:.3e} (bar {bar[b]:.1e}; SuperLU {lu_err[b]:.1e})"
                worst[b] = max(worst.get(b, 0.0), e)
        # the norms the refinement decision reads: ||b|| and ||b - A x|| of the returned x (residual as the
        # sequential CSR product forms it, bit-identical to the device's rows)
        res = r - s.A @ x
        np.testing.assert_allclose(info.rhs_norm, math.sqrt(math.fsum(r * r)), rtol=1e-12)
        np.testing.assert_allclose(info.residual_norm, math.sqrt(math.fsum(res * res)), rtol=1e-12, atol=1e-300)
    return worst, seen


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_preconditioner_is_the_exact_inverse_on_trees(case):
    """z = P^{-1} r equals A^{-1} r on trees, block by block, for r = random flux rows only, pressure rows only,
    multiplier rows only (nodal pressure rows only, continuous pressure) and all rows.

    Bar per block, relative to the block's norm: max(1e-13, 100 x the error of float64 SuperLU on the same r,
    10 eps L), L the longest chain of dependent eliminations (tree depth + flux dofs along one edge).  Error analysis
    of the last term: the sweeps carry the multipliers down the tree and the back-substitution carries the pressure
    along an edge by recurrences (lam_child = r / d + gd lam_parent, p_a = p_{a-1} + r_qa - (M q)_a), one rounding
    per step; the fluxes and pressure increments are then differences of those accumulated values, so their relative
    error grows like eps times the path length.  SuperLU's fill-reducing order has no such chains.  It matters only
    for deep chains and long edges (the 398-level chain: 1.4e-13 observed; P3/P2 with 40 cells per edge: 1.3e-13);
    for L <= 45 the 1e-13 floor is the larger term.  A wrong or missing operator term is orders of magnitude above."""
    name, build, N, (fd, pd), chunk_nodes, extra, launches = case
    s = System(build(), N, fd, pd, chunk_nodes=chunk_nodes, extra_R=extra, seed=len(name))
    assert s.schedule.is_forest
    if chunk_nodes is not None:
        assert s.schedule.n_chunks >= 2
    if name.startswith("chain_global"):
        levels = np.diff(s.schedule.chunk_lptr)
        assert levels.min() > 64 and s.schedule.n_chunks == 2  # no chunk fits the shared-memory sweeps
    kinds = ["flux", "pressure", "multipliers", "all"] + (["nodal"] if pd >= 1 else [])
    if s.blocks["multipliers"][1] == s.blocks["multipliers"][0]:
        kinds.remove("multipliers")
    worst, seen = _check_pc(s, kinds, seed0=17 * len(name))
    assert seen == {launches}, f"launch counts (setup, apply, fresh solve) {seen}, expected {launches}: another branch ran"
    print(f"{name}: n = {s.n}, worst block errors {worst}")


def test_preconditioner_badly_scaled_resistances():
    """R = 10^U(-4, 4) per cell.  Floor 1e-11 instead of 1e-13, error analysis: the elimination of the tree computes
    the nodes' Schur diagonals as d = diag0 - sum_c g_c^2 / d_c; where a stiff edge (large g) sits above soft ones,
    d_c is barely larger than g_c and the subtraction cancels up to log10(g_max / g_min) ~ 8 digits of that node's
    effective conductance.  SuperLU pivots on the whole saddle-point matrix and does not see this (2e-16 on these r);
    the tree elimination is observed at 7.8e-13 (N = 1, flux rows, pressure block).  A wrong operator term is O(1)."""
    G = ng.make_tree(9, 4, 5)
    rng = np.random.default_rng(5)
    for N in (1, 2):
        R = 10.0 ** rng.uniform(-4, 4, G.number_of_edges() * N)
        s = System(G, N, R=R, seed=N)
        worst, seen = _check_pc(s, ["flux", "pressure", "multipliers", "all"], seed0=40 + N, floor=1e-11)
        assert seen == {(1, 3, 5) if N == 1 else (3, 4, 8)}, seen
        print(f"badly scaled N={N}: worst block errors {worst}")


# ---- FGMRES against GMRES(m) in extended precision ---------------------------------------------------------------
def _parse_history(hist, m, its, tol):
    """ksp.history = [beta_0, est_1 .. est_m, beta_1, est_{m+1} ..., beta_final]: the restart entries by cycle and
    the Arnoldi estimates |g_{k+1}| by iteration k = 1 .. its.  A cycle ends early at an estimate <= tol."""
    beta, est = [], {}
    i, k = 0, 0
    while i < len(hist):
        beta.append(hist[i])
        i += 1
        if k >= its:
            break
        for _ in range(min(m, its - k)):
            k += 1
            est[k] = hist[i]
            i += 1
            if est[k] <= tol:
                break
    assert i == len(hist) and k == its, (len(hist), i, k, its)
    return np.asarray(beta), est


FGMRES_SIZES = [  # below one 256-row tile, a few thousand rows, above sm_count x 8 x 256 (grid-stride loops)
    ("y_n8", lambda: ng.make_tree(2, 1, 3), 8, 60),
    ("tree7_n2", lambda: ng.make_tree(7, 3, 4), 2, 60),
    ("tree10_n3", lambda: ng.make_tree(10, 3, 4, as_arrays=True), 3, 60),
]


def _check_fgmres(G, N, pc, m, max_it, seed):
    s = System(G, N, seed=seed)
    s.solver.ksp.options = {"ksp_type": "gmres", "pc_type": pc, "ksp_gmres_restart": m, "ksp_max_it": max_it,
                            "ksp_rtol": 1e-12}
    s.solver.b.array[:] = np.random.default_rng(seed).normal(size=s.n)  # every row populated
    s.solver.solve()
    its = s.solver.ksp.getIterationNumber()
    hist = list(s.solver.ksp.history)
    b, x = s.solver.b.array_r.copy(), s.solver.x.array_r.copy()
    assert len(hist) < _lib.HISTORY_LEN
    nb = float(np.linalg.norm(b))
    minv = None
    if pc == "jacobi":
        minv = np.ones(s.n, dtype=np.longdouble)
        nq = s.blocks["flux"][1]
        minv[:nq] = 1 / s.A.diagonal()[:nq].astype(np.longdouble)
    rho, beta_ref, x_ref = rp.OracleNetwork.gmres_reference(s.A, b, minv, m, its)
    rho = rho.astype(np.float64)
    beta_dev, est = _parse_history(hist, m, its, 1e-12 * s.solver.info.rhs_norm)
    worst = 0.0
    for k, e in est.items():
        if rho[k] > 1e-9 * nb:
            assert abs(e - rho[k]) <= 1e-10 * nb, f"iteration {k}: estimate {e:.6e}, reference {rho[k]:.6e}"
            worst = max(worst, abs(e - rho[k]) / nb)
    for c, (bt, ref) in enumerate(zip(beta_dev, beta_ref.astype(np.float64))):
        if ref > 1e-9 * nb:
            assert abs(bt - ref) <= 1e-8 * ref, f"restart {c}: true residual {bt:.6e}, reference {ref:.6e}"
    res = b.astype(np.longdouble) - s.A.astype(np.longdouble) @ x.astype(np.longdouble)
    true_res = float(np.sqrt(np.sum(res * res)))
    if rho[its] > 1e-9 * nb:
        assert abs(true_res - rho[its]) <= 1e-8 * rho[its], (true_res, rho[its])
    else:
        assert true_res <= 1e-9 * nb
    return its, worst


@pytest.mark.parametrize("m", [1, 7, 8, 9, 17, 30])
@pytest.mark.parametrize("pc", ["none", "jacobi"])
@pytest.mark.parametrize("size", FGMRES_SIZES, ids=[c[0] for c in FGMRES_SIZES])
def test_fgmres_history_matches_extended_precision_gmres(size, pc, m):
    """The Arnoldi estimates |g_{k+1}| of ksp.history are GMRES(m)'s minimal residuals to 1e-10 ||b|| while those
    exceed 1e-9 ||b||; the restart entries and the returned x's exact residual agree with the reference to 1e-8.
    Restart lengths 1 .. 30 run multi_dot / multi_axpy with K = 1 .. 8 and chunked over 8."""
    name, build, N, max_it = size
    its, worst = _check_fgmres(build(), N, pc, m, max_it, seed=m)
    assert its > min(m, 7)
    print(f"{name} pc={pc} m={m}: {its} iterations, worst |est - rho| / ||b|| = {worst:.2e}")


def test_fgmres_history_above_the_grid_stride():
    """~390 k rows (make_tree(16), N = 2): more rows than sm_count x 8 x 256, so every vector kernel's grid-stride
    loop takes several turns; restart 9 (one chunk of 8 + one of 1)."""
    its, worst = _check_fgmres(ng.make_tree(16, 16, 16, as_arrays=True), 2, "jacobi", 9, 20, seed=3)
    assert its == 20
    print(f"make_tree(16) N=2: worst |est - rho| / ||b|| = {worst:.2e}")


# ---- residual and norms -------------------------------------------------------------------------------------------
RESIDUAL_SIZES = [  # (graph, N, n_dofs): n_dofs = 0, 1, 255 (mod 256), and many tiles
    (lambda: ng.make_tree(2, 1, 3), 42, 256),
    (lambda: ng.make_tree(2, 1, 3), 170, 1024),
    (lambda: helpers.linear_graph(44, dim=3), 2, 257),
    (lambda: helpers.linear_graph(172, dim=3), 2, 1025),
    (lambda: helpers.linear_graph(65, dim=3), 1, 255),
    (lambda: helpers.linear_graph(129, dim=3), 1, 511),
    (lambda: ng.make_tree(12, 3, 4, as_arrays=True), 3, None),
]


@pytest.mark.parametrize("idx", range(len(RESIDUAL_SIZES)))
def test_residual_and_its_norm(idx):
    """nxfx_residual: r = b - A x bit-identical to the sequential CSR product, every row written (r pre-filled
    with NaN), and ||r||^2 equal to the exactly rounded sum of squares to 1e-12."""
    build, N, n_expected = RESIDUAL_SIZES[idx]
    s = System(build(), N, seed=idx)
    if n_expected is not None:
        assert s.n == n_expected
    rng = np.random.default_rng(idx)
    for scale in (1.0, 1e-8):
        x, b = rng.normal(size=s.n), rng.normal(size=s.n)
        b = s.A @ x + scale * b  # scale 1e-8: a small residual with cancellation in every row
        xd, bd, rd = s.dev.from_host(x), s.dev.from_host(b), s.dev.from_host(np.full(s.n, np.nan))
        s.solver.A.bind()
        nrm2 = C.c_double()
        s.dev.call("nxfx_residual", bd.c_ptr, xd.c_ptr, rd.c_ptr, C.byref(nrm2))
        r = rd.download()
        ref = b - s.A @ x
        assert np.array_equal(r, ref), f"{np.count_nonzero(r != ref)} rows differ from b - A x"
        np.testing.assert_allclose(nrm2.value, math.fsum(ref * ref), rtol=1e-12)
