"""Convenience functions for post-processing (drop-in for ``networks_fenicsx.post_processing``,
post_processing.py:19-97)."""

from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from .assembly import _is_cuda_tensor
from .fem import Function, FunctionSpace
from .mesh import NetworkMesh

__all__ = ["extract_global_flux", "export_functions", "export_submeshes"]


def extract_global_flux(graph_mesh: NetworkMesh, functions: list[Function]) -> Function:
    """Gather the per-colour fluxes into one DG function on the parent mesh
    (post_processing.py:19-52): cell ``c`` holds the flux at its first and second vertex.

    Args:
        graph_mesh: The network mesh
        functions: The list of functions ``[flux_1, ..., flux_M, pressure, lm]``; functions of
            ``Solver.create_functions(device=True)`` (or any functions whose arrays are CUDA tensors) give a
            function whose ``x.array`` is a CUDA tensor (no host copy; ready for the current torch stream)
    """
    flux_functions = functions[:-2]
    q_degree = flux_functions[0].function_space.element.basix_element.degree
    nc = graph_mesh.mesh.topology.index_map(1).size_local
    V = FunctionSpace(
        graph_mesh.mesh, q_degree, True, (q_degree + 1) * nc, 0,
        lambda: np.arange((q_degree + 1) * nc, dtype=np.int32).reshape(nc, q_degree + 1), "global_flux",
    )
    dev = graph_mesh.device
    if _is_cuda_tensor(flux_functions[0].x.array):
        return _global_flux_device(graph_mesh, flux_functions, V, q_degree)
    if q_degree != 1:
        # higher order: host gather through the cell -> dof tables of the per-colour spaces
        global_q = Function(V, name="Global_Flux")
        out = global_q.x.array.reshape(nc, q_degree + 1)
        for i, flux in enumerate(flux_functions):
            flux.name = f"Flux_{i}"
            cells = graph_mesh.entity_maps[i].sub_topology_to_topology(
                np.arange(flux.function_space.dofmap.list.shape[0], dtype=np.int32))
            out[cells] = flux.x.array[flux.function_space.dofmap.list]
        return global_q
    global_q = Function(V, name="Global_Flux", array=dev.pinned(V.num_dofs))
    nq = sum(f.x.array.size for f in flux_functions)
    xq = dev.empty(nq)
    off = 0
    for i, flux in enumerate(flux_functions):
        flux.name = f"Flux_{i}"
        n = flux.x.array.size
        dev.call("nxfx_memcpy_h2d", C.c_void_p(xq.ptr + 8 * off), C.c_void_p(flux.x.array.ctypes.data), C.c_size_t(8 * n))
        off += n
    out = dev.empty(V.num_dofs)
    dev.call("nxfx_global_flux", xq.c_ptr, out.c_ptr)
    out.download(global_q.x.array)
    return global_q


def _global_flux_device(graph_mesh: NetworkMesh, flux_functions: list[Function], V: FunctionSpace,
                        q_degree: int) -> Function:
    """``extract_global_flux`` of device functions: P1 through ``nxfx_global_flux``, higher degrees through
    ``nxfx_gather`` over the DG entry -> flux dof table (the host gather below, built once per mesh and degree).
    The output (and the scratch copy of flux blocks that are not contiguous) come from torch's caching allocator,
    so that a time loop calling this allocates and frees nothing through the driver (no implicit host waits)."""
    import torch  # noqa: PLC0415

    dev = graph_mesh.device
    arrays = [f.x.array for f in flux_functions]
    for i, flux in enumerate(flux_functions):
        flux.name = f"Flux_{i}"
    cuda = torch.device("cuda", dev.index)
    out = torch.empty(V.num_dofs, dtype=torch.float64, device=cuda)
    # the flux blocks of create_functions(device=True) follow each other in one buffer: read them in place
    src = arrays[0].data_ptr()
    xq = None
    if any(a.data_ptr() != src + 8 * sum(b.numel() for b in arrays[:i]) for i, a in enumerate(arrays)):
        xq = torch.empty(sum(a.numel() for a in arrays), dtype=torch.float64, device=cuda)
        src = xq.data_ptr()
    dev.wait_for_torch(*[t for t in (out, xq) if t is not None])
    if xq is not None:
        off = 0
        for a in arrays:
            if a.numel():
                dev.call("nxfx_memcpy_d2d", C.c_void_p(src + 8 * off), C.c_void_p(a.data_ptr()),
                         C.c_size_t(8 * a.numel()))
            off += a.numel()
    out_ptr = C.c_void_p(out.data_ptr())
    if q_degree == 1:
        dev.call("nxfx_global_flux", C.c_void_p(src), out_ptr)
    else:
        if getattr(graph_mesh, "_global_flux_index", None) is None:
            graph_mesh._global_flux_index = {}
        cache = graph_mesh._global_flux_index
        if q_degree not in cache:
            nc = V.num_dofs // (q_degree + 1)
            idx = np.zeros((nc, q_degree + 1), dtype=np.int32)
            off = 0
            for i, flux in enumerate(flux_functions):
                dm = flux.function_space.dofmap.list
                cells = graph_mesh.entity_maps[i].sub_topology_to_topology(np.arange(dm.shape[0], dtype=np.int32))
                idx[cells] = off + dm
                off += flux.function_space.num_dofs
            cache[q_degree] = dev.from_host(idx.ravel())
        dev.call("nxfx_gather", C.c_void_p(src), cache[q_degree].c_ptr, 1, V.num_dofs, 1, out_ptr)
    global_q = Function(V, name="Global_Flux", array=out)
    dev.torch_wait()
    return global_q


def export_functions(functions: list[Function], outpath: Path | str):
    """Write the solution functions as ``.npy`` arrays (``flux_i``, ``pressure``, ``lm``) --
    the reference writes ADIOS2 VTX files (post_processing.py:55-78); ADIOS2 is not part of this
    build, see DESIGN.md "out of scope".  Device functions are copied to the host."""
    export_path = Path(outpath)
    export_path.mkdir(parents=True, exist_ok=True)
    for i, q in enumerate(functions[:-2]):
        np.save(export_path / f"flux_{i}.npy", _host(q.x.array))
    np.save(export_path / "pressure.npy", _host(functions[-2].x.array))
    np.save(export_path / "lm.npy", _host(functions[-1].x.array))


def _host(a) -> np.ndarray:
    return a.cpu().numpy() if _is_cuda_tensor(a) else a


def export_submeshes(network_mesh: NetworkMesh, outpath: str | Path):
    """Write each colour submesh (vertices, cells, facet markers) as ``.npz``
    (reference: XDMF, post_processing.py:81-97)."""
    outpath = Path(outpath)
    outpath.mkdir(parents=True, exist_ok=True)
    for i in range(network_mesh.num_edge_colors):
        sm = network_mesh.submeshes[i]
        tags = network_mesh.submesh_facet_markers[i]
        np.savez(
            outpath / f"submesh_{i}.npz", x=sm.geometry.x,
            cells=sm.topology.connectivity(1, 0).array.reshape(-1, 2),
            facet_indices=tags.indices, facet_values=tags.values,
        )
