"""The pipelined CSR product (spmv_pipe_kernel) where the parity and operator tests do not reach it.

* many tiles per block: each block's ring of tiles is refilled and wraps around many times;
* rows longer than the entries a thread keeps in registers (a hub of degree 12 with N = 1): those rows are
  summed straight from the ring;
* tiles whose rows straddle the flux / pressure / multiplier block boundaries;
* the norms-only pass inside nxfx_solve against the pass that writes r: the norm the solve reports is the norm
  nxfx_residual returns for the same b and x, and the correction of a forced refinement is P^{-1}(b - A x).

Every row is compared with SciPy's sequential CSR product bit for bit.
"""

import ctypes as C
import math

import networkx as nx
import numpy as np
import pytest

from networks_fenicsx_b200 import _lib
from networks_fenicsx_b200 import network_generation as ng
from tests.test_gpu_operators import System

pytestmark = pytest.mark.gpu

TILE_ROWS = 256


def _hub_graph(degree=12):
    """inlet -> hub -> `degree` leaves, in 3D: the hub's rows hold more than 8 entries."""
    G = nx.DiGraph()
    G.add_node(0, pos=np.array([0.0, 0.0, -1.0]))
    G.add_node(1, pos=np.zeros(3))
    G.add_edge(0, 1)
    for k in range(degree):
        a = 2.0 * np.pi * k / degree
        G.add_node(2 + k, pos=np.array([np.cos(a), np.sin(a), 0.5 + 0.1 * k]))
        G.add_edge(1, 2 + k)
    return G


CASES = {
    "many_ring_turns": (lambda: ng.make_tree(19, 19, 19, as_arrays=True), 1),
    "long_rows": (lambda: _hub_graph(12), 1),
    "long_rows_refined": (lambda: _hub_graph(40), 3),
}


@pytest.fixture(scope="module", params=list(CASES))
def system(request):
    build, N = CASES[request.param]
    s = System(build(), N, seed=7)
    s.case = request.param
    return s


def test_shape_reaches_the_path(system):
    s = system
    lens = np.diff(s.A.indptr)
    if s.case == "many_ring_turns":
        assert s.n // TILE_ROWS >= 8 * 148 * 3, "fewer than 8 tiles per block of a B200 grid (3 blocks per SM)"
        bounds = [s.blocks["pressure"][0], s.blocks["multipliers"][0]]
        assert any(b % TILE_ROWS for b in bounds), "no tile straddles a block boundary"
    else:
        assert lens.max() > 8, f"longest row {lens.max()}"


def test_spmv_and_residual_rows(system):
    s = system
    s.solver.A.bind()
    rng = np.random.default_rng(3)
    x, b = rng.normal(size=s.n), rng.normal(size=s.n)
    xd, bd = s.dev.from_host(x), s.dev.from_host(b)
    yd, rd = s.dev.from_host(np.full(s.n, np.nan)), s.dev.from_host(np.full(s.n, np.nan))
    s.dev.call("nxfx_spmv", xd.c_ptr, yd.c_ptr)
    ax = s.A @ x
    y = yd.download()
    assert np.array_equal(y, ax), f"{np.count_nonzero(y != ax)} rows of A x differ"
    nrm2 = C.c_double()
    s.dev.call("nxfx_residual", bd.c_ptr, xd.c_ptr, rd.c_ptr, C.byref(nrm2))
    ref = b - ax
    r = rd.download()
    assert np.array_equal(r, ref), f"{np.count_nonzero(r != ref)} rows of b - A x differ"
    np.testing.assert_allclose(nrm2.value, math.fsum(ref * ref), rtol=1e-12)


def _solve(s, b, refine_steps, refine_rtol):
    """A freshly assembled matrix, then nxfx_solve (preonly) with a final residual of the returned x."""
    s.assemble()
    o = s.solver.ksp.options
    o.update({"nxfx_refine_steps": refine_steps, "nxfx_refine_rtol": refine_rtol, "nxfx_final_residual": True})
    opts = s.solver.solve_options()
    info = _lib.SolveInfo()
    bd, xd = s.dev.from_host(b), s.dev.from_host(np.full(s.n, np.nan))
    s.dev.call("nxfx_solve", bd.c_ptr, xd.c_ptr, C.byref(opts), C.byref(info))
    return xd.download(), info


def _residual(s, b, x):
    s.solver.A.bind()
    bd, xd, rd = s.dev.from_host(b), s.dev.from_host(x), s.dev.from_host(np.full(s.n, np.nan))
    nrm2 = C.c_double()
    s.dev.call("nxfx_residual", bd.c_ptr, xd.c_ptr, rd.c_ptr, C.byref(nrm2))
    r = rd.download()
    ref = b - s.A @ x
    assert np.array_equal(r, ref), f"{np.count_nonzero(r != ref)} rows of b - A x differ"
    return r, nrm2.value


def test_norms_only_pass_equals_written_pass(system):
    s = system
    b = np.random.default_rng(5).normal(size=s.n)
    # no refinement: the reported norm comes from the norms-only pass on the returned x
    x0, info0 = _solve(s, b, 0, 0.0)
    r0, n2 = _residual(s, b, x0)
    assert info0.residual_norm == math.sqrt(n2)
    # a forced refinement: the norms-only pass on x0, the written pass, the correction, the check of x1
    x1, info1 = _solve(s, b, 1, 0.0)
    assert info1.iterations == 2
    assert info1.history_len >= 2 and info1.history[0] == info0.residual_norm
    _, n2_1 = _residual(s, b, x1)
    assert info1.residual_norm == math.sqrt(n2_1)
    # the correction is P^{-1} of the written residual rows (which equal b - A x0 above)
    s.solver.A.bind()
    rd, zd = s.dev.from_host(r0), s.dev.from_host(np.full(s.n, np.nan))
    s.dev.call("nxfx_pc_setup")
    s.dev.call("nxfx_pc_apply", rd.c_ptr, zd.c_ptr)
    z = zd.download()
    np.testing.assert_allclose(x1 - x0, z, rtol=1e-9, atol=1e-12 * np.abs(x0).max())
