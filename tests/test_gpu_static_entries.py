"""Re-assembly without ADD_VALUES writes only the flux rows of the matrix: the pressure rows {-1, +1} and the
multiplier rows (0, +1) / (-1, 0) depend on the pattern alone and stay from the previous assembly
(``MatState::static_valid``).  After every sequence below the matrix values and the right-hand side are
compared bit for bit with the first assembly of a fresh matrix on the same forms, and the flag is checked
after every call that must clear it."""

import ctypes as C

import numpy as np
import pytest

import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200 import network_generation as ng

pytestmark = pytest.mark.gpu

P_Y = lambda x: x[1]  # noqa: E731
P_X = lambda x: 2.0 * x[0] - x[2]  # noqa: E731


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def fresh(asm):
    """Values and rhs of the first assembly of a new matrix and vector on the assembler's current forms."""
    A, b = asm.assemble()
    assert A.accumulated == 1
    out = bits(A.getValuesCSR()[2]).copy(), bits(b.array_r).copy()
    del A, b
    return out


def check(solver, ref):
    va, bv = ref
    assert np.array_equal(bits(solver.A.getValuesCSR()[2]), va), "matrix values differ from a fresh assembly"
    assert np.array_equal(bits(solver.b.array_r), bv), "right-hand side differs from a fresh assembly"


def coefficients(nm, seed):
    rng = np.random.default_rng(seed)
    nc = nm.mesh.topology.index_map(1).size_local
    return rng.uniform(0.5, 2.0, nc), rng.normal(size=nc)


def setup(N, seed=0, G=None):
    nm = nxfx.NetworkMesh(G if G is not None else ng.make_tree(7, 3, 4), N=N, color_strategy="smallest_last")
    asm = nxfx.HydraulicNetworkAssembler(nm)
    R, f = coefficients(nm, seed)
    asm.compute_forms(p_bc_ex=P_Y, R=R, f=f)
    return nm, asm, nxfx.Solver(asm)


def pressure_and_multiplier_slice(solver):
    rp = solver.A.pattern()[0]
    nq = sum(solver.assembler.block_sizes[:-2])
    return slice(int(rp[nq]), int(rp[-1]))


@pytest.mark.parametrize("N", [1, 3])
def test_repeated_assembly_with_changing_data(N):
    nm, asm, solver = setup(N)
    assert not solver.A.static_valid  # a new matrix
    solver.assemble()
    assert solver.A.static_valid
    for k, p_bc in enumerate((P_X, P_Y, P_X)):
        R, f = coefficients(nm, 10 + k)
        asm.compute_forms(p_bc_ex=p_bc, R=R if k != 1 else 3.5, f=f if k != 2 else 0.0)
        solver.assemble()  # skips the pressure / multiplier rows
        assert solver.A.static_valid
        check(solver, fresh(asm))
        solver.solve()


@pytest.mark.parametrize("N", [1, 3])
def test_accumulated_then_zeroed(N):
    nm, asm, solver = setup(N)
    solver.assemble()
    for k in range(2):  # ADD_VALUES: k * {-1, +1} in the pressure rows
        R, _ = coefficients(nm, 20 + k)
        asm.compute_forms(p_bc_ex=P_Y, R=R)
        asm.assemble(solver.A, solver.b)
        assert not solver.A.static_valid
        assert solver.A.accumulated == k + 2
    solver.assemble()  # zeroEntries + assemble: must rewrite every entry
    assert solver.A.static_valid and solver.A.accumulated == 1
    check(solver, fresh(asm))
    solver.assemble()
    check(solver, fresh(asm))


@pytest.mark.parametrize("N", [1, 3])
def test_zero_now_then_assemble(N):
    nm, asm, solver = setup(N)
    solver.assemble()
    solver.A.zero_now()
    assert not solver.A.static_valid
    assert not np.any(solver.A.values.download())
    solver.assemble()
    assert solver.A.static_valid
    check(solver, fresh(asm))


@pytest.mark.parametrize("N", [1, 3])
def test_rhs_only(N):
    nm, asm, solver = setup(N)
    solver.assemble()
    R, f = coefficients(nm, 30)
    asm.compute_forms(p_bc_ex=P_X, R=R, f=f)
    solver.assemble(lhs=False)  # the values keep the old R; the flag stays
    assert solver.A.static_valid
    va_old = bits(solver.A.getValuesCSR()[2]).copy()
    ref = fresh(asm)
    assert np.array_equal(bits(solver.b.array_r), ref[1])
    solver.assemble(lhs=False)
    assert np.array_equal(bits(solver.A.getValuesCSR()[2]), va_old)
    solver.assemble()
    check(solver, ref)


@pytest.mark.parametrize("N", [1, 3])
def test_two_solvers_on_one_mesh(N):
    nm, asm1, s1 = setup(N, seed=1)
    asm2 = nxfx.HydraulicNetworkAssembler(nm)
    R2, f2 = coefficients(nm, 2)
    asm2.compute_forms(p_bc_ex=P_X, R=R2, f=f2)
    s2 = nxfx.Solver(asm2)
    s1.assemble()
    s2.assemble()
    s2.A.zero_now()  # clears s2's flag only
    assert s1.A.static_valid and not s2.A.static_valid
    for _ in range(2):
        s1.assemble()
        s2.assemble()
        check(s2, fresh(asm2))
        check(s1, fresh(asm1))
        assert s1.A.static_valid and s2.A.static_valid


@pytest.mark.parametrize("N", [1, 3])
def test_writes_through_values(N):
    nm, asm, solver = setup(N)
    solver.assemble()
    ref = fresh(asm)
    sl = pressure_and_multiplier_slice(solver)
    junk = np.full(solver.A.nnz, 7.25)
    # DeviceArray writes tell the library themselves
    solver.A.values.upload(junk)
    assert not solver.A.static_valid
    solver.assemble()
    check(solver, ref)
    solver.A.values.view(sl.start, sl.stop - sl.start).zero()
    assert not solver.A.static_valid
    solver.assemble()
    check(solver, ref)
    # a raw write through the device pointer is followed by Mat.touch (nxfx_matrix_touch) ...
    dev = nm.device
    dev.call("nxfx_memset", C.c_void_p(solver.A.values.ptr), 0x3F, C.c_size_t(solver.A.values.nbytes))
    solver.A.touch()
    assert not solver.A.static_valid
    solver.assemble()
    check(solver, ref)
    # ... without it the re-assembly leaves those rows as they were: only the flux rows are written
    dev.call("nxfx_memset", C.c_void_p(solver.A.values.ptr), 0, C.c_size_t(solver.A.values.nbytes))
    solver.assemble()
    va = solver.A.getValuesCSR()[2]
    assert not np.any(va[sl])
    assert np.array_equal(bits(va[: sl.start]), ref[0][: sl.start])
    solver.A.touch()
    solver.assemble()
    check(solver, ref)


def test_higher_order_keeps_the_flag_clear():
    nm = nxfx.NetworkMesh(ng.make_tree(5, 3, 4), N=2)
    asm = nxfx.HydraulicNetworkAssembler(nm, flux_degree=2, pressure_degree=1)
    asm.compute_forms(p_bc_ex=P_Y)
    solver = nxfx.Solver(asm)
    for _ in range(2):
        solver.assemble()
        assert not solver.A.static_valid
    check(solver, fresh(asm))


def test_partitioned_in_one_process():
    G = ng.make_tree(11, 11, 11, as_arrays=True)

    def fresh_rank(s):
        return fresh(s.assembler)

    def state(s):
        return (bits(s.solver.A.getValuesCSR()[2]).copy(), bits(s.solver.b.array_r).copy(),
                s.solver.A.static_valid)

    with nxfx.PartitionedSolver(G, 1, P_Y, devices=[0, 0], chunk_nodes=64) as ps:
        ps.assemble()
        ps.solve()
        first = ps.map(fresh_rank)
        for _ in range(2):
            ps.assemble()
            got = ps.map(state)
            for (va, bv, ok), (rva, rbv) in zip(got, first):
                assert ok
                assert np.array_equal(va, rva) and np.array_equal(bv, rbv)
            hist = ps.solve(final_residual=True)
            assert hist[-1] < 1e-12, hist
        ps.map(lambda s: s.solver.A.zero_now())
        assert ps.map(lambda s: s.solver.A.static_valid) == [False, False]
        ps.assemble()
        got = ps.map(state)
        assert all(ok for _, _, ok in got)
        assert all(np.array_equal(va, rva) and np.array_equal(bv, rbv) for (va, bv, _), (rva, rbv) in zip(got, first))
