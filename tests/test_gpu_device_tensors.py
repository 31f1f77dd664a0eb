"""CUDA tensors in and out of the public API: ``compute_forms`` with device p_bc / R / f,
``NetworkMesh.vertex_coordinates_device``, ``Solver.create_functions(device=True)`` and the device
``extract_global_flux``.  The device path must reproduce the NumPy path bit for bit, move nothing over PCIe
in a time loop, and order itself against torch streams with events."""

import types

import networkx as nx
import numpy as np
import pytest

import networks_fenicsx_b200 as nxfx
from networks_fenicsx_b200 import network_generation as ng

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _build(G, N, strategy, degrees):
    nm = nxfx.NetworkMesh(G, N=N, color_strategy=strategy)
    return nm, nxfx.HydraulicNetworkAssembler(nm, *degrees)


def _host_run(G, N, strategy, degrees, comp, R, f):
    nm, asm = _build(G, N, strategy, degrees)
    pbc = np.ascontiguousarray(nm.mesh.geometry.x[:, comp])
    asm.compute_forms(p_bc_ex=pbc, R=R, f=f)
    solver = nxfx.Solver(asm)
    solver.assemble()
    sol = solver.solve()
    return solver, sol


def _device_run(G, N, strategy, degrees, comp, R, f):
    nm, asm = _build(G, N, strategy, degrees)
    X = nm.vertex_coordinates_device()
    assert X.shape == (nm.mesh.geometry.x.shape[0], 3) and X.stride() == (4, 1)
    assert torch.equal(X.cpu(), torch.from_numpy(nm.mesh.geometry.x))  # a view of the records, no copy
    to_dev = lambda c: _cuda(c) if isinstance(c, np.ndarray) else c  # noqa: E731
    asm.compute_forms(p_bc_ex=X[:, comp].contiguous(), R=to_dev(R), f=to_dev(f))
    solver = nxfx.Solver(asm)
    solver.assemble()
    fns = solver.create_functions(device=True)
    assert all(fn.x.array.is_cuda for fn in fns)
    out = solver.solve(fns)
    assert out is fns
    return solver, fns


def _same_system_and_solution(host, dev):
    (hs, hsol), (ds, dfns) = host, dev
    for a, b in zip(hs.A.getValuesCSR(), ds.A.getValuesCSR()):
        assert np.array_equal(a, b)
    assert np.array_equal(hs.b.array_r, ds.b.array_r)
    x_host = np.concatenate([fn.x.array for fn in hsol])
    x_dev = torch.cat([fn.x.array for fn in dfns]).cpu().numpy()
    assert np.array_equal(x_host, x_dev)
    assert np.array_equal(ds.x.array_r, x_dev)  # solver.x holds the same values


def test_device_inputs_and_functions_match_the_numpy_path():
    rng = np.random.default_rng(7)
    cases = []
    G = ng.make_tree(6, 6, 6)
    E = G.number_of_edges()
    for N in (1, 3):
        cases.append((G, N, "smallest_last", (1, 0), 1, rng.uniform(0.5, 2.0, E * N), rng.normal(size=E * N)))
    cases.append((G, 3, "smallest_last", (1, 0), 0, rng.uniform(0.5, 2.0, E), None))  # per-edge R
    Ga = ng.make_arterial_tree(N=5, direction=np.array([0.1, 1.0, 0.0]))
    radius = np.array([Ga.edges[e]["radius"] for e in Ga.edges()])
    Na = 8
    cases.append((Ga, Na, nx.coloring.strategy_largest_first, (1, 0), 1, 8.0 * 1.0 / (np.pi * radius**4),
                  rng.normal(size=Ga.number_of_edges() * Na)))
    Gh = ng.make_tree(4, 4, 4)
    Eh = Gh.number_of_edges()
    for degrees in ((2, 1), (2, 0)):
        cases.append((Gh, 2, "smallest_last", degrees, 1, rng.uniform(0.5, 2.0, Eh), rng.normal(size=2 * Eh)))
    for G_, N, strategy, degrees, comp, R, f in cases:
        _same_system_and_solution(_host_run(G_, N, strategy, degrees, comp, R, f),
                                  _device_run(G_, N, strategy, degrees, comp, R, f))


def test_second_assembler_on_the_mesh_restores_the_device_boundary_pressure():
    G = ng.make_tree(5, 5, 5)
    host = _host_run(G, 2, "smallest_last", (1, 0), 1, None, None)
    nm = nxfx.NetworkMesh(G, N=2, color_strategy="smallest_last")
    X = nm.vertex_coordinates_device()
    a1 = nxfx.HydraulicNetworkAssembler(nm)
    a1.compute_forms(p_bc_ex=X[:, 1].contiguous())
    s1 = nxfx.Solver(a1)
    a2 = nxfx.HydraulicNetworkAssembler(nm)
    a2.compute_forms(p_bc_ex=(3.0 * X[:, 0] + 1.0).contiguous())  # overwrites the vertex records
    s1.assemble()  # restores a1's p_bc from its own device copy
    fns = s1.create_functions(device=True)
    _same_system_and_solution(host, (s1, s1.solve(fns)))


def test_whole_network_device_coefficients_are_restricted_to_the_rank():
    G = ng.make_tree(9, 9, 9, as_arrays=True)
    E, N = G.number_of_edges(), 2
    rng = np.random.default_rng(3)
    R_edge, f_cell = rng.uniform(0.5, 2.0, E), rng.normal(size=E * N)
    for rank in range(2):
        comm = types.SimpleNamespace(size=2, rank=rank)
        nm = nxfx.NetworkMesh(G, N=N, color_strategy="smallest_last", comm=comm, device=0)
        assert nm._partition is not None and nm.graph_edges.shape[0] < E
        asm = nxfx.HydraulicNetworkAssembler(nm)
        asm.compute_forms(p_bc_ex=lambda x: x[1], R=R_edge, f=f_cell)
        R_ref, f_ref = asm._R[0].download(), asm._f[0].download()
        asm.compute_forms(p_bc_ex=lambda x: x[1], R=_cuda(R_edge), f=_cuda(f_cell))
        assert np.array_equal(asm._R[0].download(), R_ref)
        assert np.array_equal(asm._f[0].download(), f_ref)
        # the whole network per cell / the local edges per edge take the same route as the NumPy arrays
        asm.compute_forms(p_bc_ex=lambda x: x[1], R=_cuda(np.repeat(R_edge, N)), f=_cuda(f_ref))
        assert np.array_equal(asm._R[0].download(), R_ref)
        assert np.array_equal(asm._f[0].download(), f_ref)


class _CallLog:
    def __init__(self, dev):
        self.names, self._call = [], dev.call
        dev.call = self

    def __call__(self, name, *args):
        self.names.append(name)
        return self._call(name, *args)


def test_a_device_time_loop_moves_nothing_over_pcie():
    G = ng.make_tree(8, 8, 8)
    rng = np.random.default_rng(0)
    R = rng.uniform(0.5, 2.0, G.number_of_edges())
    host_calls = {}
    for device in (False, True):
        nm = nxfx.NetworkMesh(G, N=1, color_strategy="smallest_last")
        asm = nxfx.HydraulicNetworkAssembler(nm)
        X = nm.vertex_coordinates_device()
        if device:
            pbc, Rc, fns_of = (lambda t: (X[:, 1] * (1.0 + t)).contiguous()), _cuda(R), True
        else:
            Xh = nm.mesh.geometry.x
            pbc, Rc, fns_of = (lambda t: Xh[:, 1] * (1.0 + t)), R, False
        asm.compute_forms(p_bc_ex=pbc(0.0), R=Rc)
        solver = nxfx.Solver(asm)
        fns = solver.create_functions(device=fns_of)

        def step(t, asm=asm, solver=solver, fns=fns, pbc=pbc, Rc=Rc):
            asm.compute_forms(p_bc_ex=pbc(t), R=Rc)
            solver.assemble()
            solver.solve(fns)

        step(0.0)  # warm-up: the symbolic phase synchronises once
        log = _CallLog(nm.device)
        step(0.5)
        host_calls[device] = log.names
    dev_calls = host_calls[True]
    assert not {"nxfx_memcpy_h2d", "nxfx_memcpy_d2h", "nxfx_sync"} & set(dev_calls), dev_calls
    assert dev_calls.count("nxfx_solve") == 1  # the one host wait of the step
    # the host path of the same loop uploads p_bc / R and waits for the device in compute_forms
    assert {"nxfx_memcpy_h2d", "nxfx_sync"} <= set(host_calls[False]), host_calls[False]


def _reference_x(G, N, pbc_host, R):
    nm = nxfx.NetworkMesh(G, N=N, color_strategy="smallest_last")
    asm = nxfx.HydraulicNetworkAssembler(nm)
    asm.compute_forms(p_bc_ex=pbc_host, R=R)
    solver = nxfx.Solver(asm)
    solver.assemble()
    return np.concatenate([fn.x.array for fn in solver.solve()])


SLEEP_CYCLES = 200_000_000  # ~0.1 s: far longer than everything the host enqueues meanwhile


def test_inputs_written_on_a_side_stream_are_read_after_that_stream():
    G = ng.make_tree(7, 7, 7)
    nm = nxfx.NetworkMesh(G, N=2, color_strategy="smallest_last")
    Xh = nm.mesh.geometry.x
    E = G.number_of_edges()
    R = np.linspace(0.5, 2.0, E)
    x_ref = _reference_x(G, 2, np.ascontiguousarray(2.0 * Xh[:, 1] - 1.0), R)
    asm = nxfx.HydraulicNetworkAssembler(nm)
    asm.compute_forms(p_bc_ex=lambda x: 0 * x[0], R=np.zeros(E))  # the device buffers exist before the timed part
    solver = nxfx.Solver(asm)
    fns = solver.create_functions(device=True)
    X = nm.vertex_coordinates_device()
    pbc = torch.zeros(X.shape[0], dtype=torch.float64, device="cuda")
    Rt = torch.zeros(E, dtype=torch.float64, device="cuda")
    R_src = _cuda(R)  # built here: a host->device copy inside the block below would wait for the side stream
    side = torch.cuda.Stream()

    def write(sleep):
        torch.cuda._sleep(sleep)
        pbc.copy_(2.0 * X[:, 1] - 1.0)
        Rt.copy_(R_src)

    with torch.cuda.stream(side):  # once untimed: the first launch of a kernel loads it, which waits for the device
        write(1)
        asm.compute_forms(p_bc_ex=pbc, R=Rt)
        solver.assemble()
        solver.solve(fns)
    torch.cuda.synchronize()
    pbc.fill_(-3.0)  # stale values: a solvable system with another solution
    Rt.fill_(1.0)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        write(SLEEP_CYCLES)
        asm.compute_forms(p_bc_ex=pbc, R=Rt)  # the library stream must wait for the writes behind the sleep
        # the library enqueued its reads while the writes were still pending: without the event it reads stale values
        assert not side.query(), "the side stream finished before compute_forms: the test would decide nothing"
        solver.assemble()
        solver.solve(fns)
        x = torch.cat([fn.x.array for fn in fns])  # on the side stream: ordered after the solve
    torch.cuda.synchronize()
    assert np.array_equal(x.cpu().numpy(), x_ref)


def test_an_input_freed_right_after_compute_forms_is_not_reused_before_it_is_read():
    G = ng.make_tree(7, 7, 7)
    nm = nxfx.NetworkMesh(G, N=1, color_strategy="smallest_last")
    Xh = nm.mesh.geometry.x
    x_ref = _reference_x(G, 1, np.ascontiguousarray(Xh[:, 1]), None)
    asm = nxfx.HydraulicNetworkAssembler(nm)
    asm.compute_forms(p_bc_ex=lambda x: 0 * x[0])
    solver = nxfx.Solver(asm)
    fns = solver.create_functions(device=True)
    X = nm.vertex_coordinates_device()
    side = torch.cuda.Stream()
    torch.cuda._sleep(1)  # the first launch of a kernel loads it, which waits for the device: not in the timed part
    with torch.cuda.stream(side):
        torch.full((X.shape[0],), 1e6, dtype=torch.float64, device="cuda")
        asm.compute_forms(p_bc_ex=X[:, 1].contiguous())
    torch.cuda.synchronize()
    asm.compute_forms(p_bc_ex=lambda x: 0 * x[0])
    torch.cuda._sleep(SLEEP_CYCLES)  # the library's (legacy default) stream is busy
    with torch.cuda.stream(side):
        pbc = X[:, 1].contiguous()  # allocated and written on the side stream
        asm.compute_forms(p_bc_ex=pbc)
        del pbc
        junk = torch.full((X.shape[0],), 1e6, dtype=torch.float64, device="cuda")  # same size, same stream
        assert not torch.cuda.default_stream().query(), "the library's stream finished early: the test would decide nothing"
        solver.assemble()
        solver.solve(fns)
        x = torch.cat([fn.x.array for fn in fns])
    torch.cuda.synchronize()
    del junk
    assert np.array_equal(x.cpu().numpy(), x_ref)


def test_device_global_flux_and_export_match_the_host_functions(tmp_path):
    G = ng.make_tree(5, 5, 5)
    for degrees, N in (((1, 0), 3), ((2, 1), 2), ((3, 2), 2)):
        nm, asm = _build(G, N, "smallest_last", degrees)
        asm.compute_forms(p_bc_ex=lambda x: x[1], f=1.0)
        solver = nxfx.Solver(asm)
        solver.assemble()
        host_fns = solver.solve()
        host = nxfx.post_processing.extract_global_flux(nm, host_fns)
        dev_fns = solver.solve(solver.create_functions(device=True))
        gq = nxfx.post_processing.extract_global_flux(nm, dev_fns)  # the first call builds the index table
        assert gq.x.array.is_cuda
        assert np.array_equal(gq.x.array.cpu().numpy(), host.x.array)
        log = _CallLog(nm.device)
        again = nxfx.post_processing.extract_global_flux(nm, dev_fns)
        del nm.device.call
        assert not {"nxfx_malloc", "nxfx_memcpy_h2d", "nxfx_memcpy_d2h", "nxfx_sync"} & set(log.names), log.names
        assert np.array_equal(again.x.array.cpu().numpy(), host.x.array)
        # functions of the caller's own tensors (not one buffer): gathered into a scratch copy first
        own = [nxfx.fem.Function(fn.function_space, name=fn.name, array=fn.x.array.clone()) for fn in dev_fns]
        assert np.array_equal(nxfx.post_processing.extract_global_flux(nm, own).x.array.cpu().numpy(), host.x.array)
        tag = f"P{degrees[0]}{degrees[1]}"
        nxfx.post_processing.export_functions(host_fns, tmp_path / f"host_{tag}")
        nxfx.post_processing.export_functions(dev_fns, tmp_path / f"dev_{tag}")
        files = sorted(p.name for p in (tmp_path / f"host_{tag}").iterdir())
        assert files == sorted(p.name for p in (tmp_path / f"dev_{tag}").iterdir())
        for name in files:
            assert np.array_equal(np.load(tmp_path / f"host_{tag}" / name), np.load(tmp_path / f"dev_{tag}" / name))


def test_invalid_device_tensors_raise_before_anything_is_launched():
    G = ng.make_tree(4, 4, 4)
    nm = nxfx.NetworkMesh(G, N=2, color_strategy="smallest_last")
    asm = nxfx.HydraulicNetworkAssembler(nm)
    X = nm.vertex_coordinates_device()
    nv, nc = X.shape[0], 2 * G.number_of_edges()
    good = X[:, 1].contiguous()
    asm.compute_forms(p_bc_ex=good)
    bad = [
        (TypeError, dict(p_bc_ex=good.float())),
        (ValueError, dict(p_bc_ex=X[:, 1])),  # a strided view
        (ValueError, dict(p_bc_ex=good[:-1])),
        (TypeError, dict(p_bc_ex=good, R=torch.ones(nc, dtype=torch.float32, device="cuda"))),
        (ValueError, dict(p_bc_ex=good, f=torch.ones(2 * nc, dtype=torch.float64, device="cuda")[::2])),
        (ValueError, dict(p_bc_ex=good, R=torch.ones(nc + 1, dtype=torch.float64, device="cuda"))),
    ]
    if torch.cuda.device_count() > 1:
        bad.append((ValueError, dict(p_bc_ex=good.to("cuda:1"))))
    for exc, kwargs in bad:
        l0 = nm.device.launch_count
        with pytest.raises(exc):
            asm.compute_forms(**kwargs)
        assert nm.device.launch_count == l0, kwargs


def test_device_functions_on_a_partitioned_network():
    """Through the distributed layer (two ranks sharing cuda:0, gloo): the local dofs are copied from solver.x
    into the device functions (tests/dist_check_device.py)."""
    import os
    import pathlib
    import subprocess
    import sys

    from tests import helpers

    root = pathlib.Path(__file__).resolve().parent.parent
    env = dict(os.environ, NXFX_DIST_ONE_GPU="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(helpers.free_port()),
           str(root / "tests" / "dist_check_device.py"), "8", "2", "2", "1"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "-> OK" in out.stdout, out.stdout[-3000:]
