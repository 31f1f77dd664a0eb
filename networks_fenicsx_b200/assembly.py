"""Assembler of the hydraulic network model (drop-in for ``networks_fenicsx.assembly``,
assembly.py:95-398).

.. math::
    R q + \\frac{\\mathrm{d}}{\\mathrm{d}s} p = 0, \\qquad \\frac{\\mathrm{d}}{\\mathrm{d}s} q = f

The UFL/FFCx/DOLFINx pipeline (assembly.py:164-299 forms, :354-367 assembly) is replaced by the
hand-written row-owned CUDA assembly kernel behind ``nxfx_assemble``; this file only keeps the
reference's Python surface, evaluates the boundary pressure at the mesh vertices
(assembly.py:225-234) and prepares the coefficient arrays.
"""

from __future__ import annotations

import ctypes as C
import logging
import sys
import typing

import numpy as np
import numpy.typing as npt

from .common import timed
from .fem import CoordinateExpr, Function, FunctionSpace
from .la import Mat, Vec
from .mesh import NetworkMesh

__all__ = ["HydraulicNetworkAssembler", "PressureFunction", "compute_integration_data"]


class PressureFunction(typing.Protocol):
    def eval(self, x: npt.NDArray[np.floating]) -> npt.NDArray[np.inexact]: ...


@timed("nxfx:compute_integration_data")
def compute_integration_data(
    network_mesh: NetworkMesh,
) -> tuple[dict[int, npt.NDArray[np.int32]], dict[int, npt.NDArray[np.int32]]]:
    """(parent cell, local facet) pairs of the bifurcation end-vertices per colour
    (assembly.py:28-92), in closed form: an edge entering a bifurcation contributes
    ``(last cell, 1)`` to the influx list of its colour, an edge leaving one contributes
    ``(first cell, 0)`` to the outflux list; pairs are in ascending parent-cell order."""
    N = network_mesh.cells_per_edge
    edges = network_mesh.graph_edges
    lm = network_mesh.node_multiplier_index
    colors = network_mesh.edge_colors
    e_in = np.flatnonzero(lm[edges[:, 1]] >= 0)
    e_out = np.flatnonzero(lm[edges[:, 0]] >= 0)
    infl: dict[int, npt.NDArray[np.int32]] = {}
    outfl: dict[int, npt.NDArray[np.int32]] = {}
    if network_mesh.num_edge_colors > 4096:  # uncoloured mode: avoid C passes over all edges
        col_in, col_out = colors[e_in], colors[e_out]
        infl = {int(c): np.empty(0, dtype=np.int32) for c in range(network_mesh.num_edge_colors)}
        outfl = {int(c): np.empty(0, dtype=np.int32) for c in range(network_mesh.num_edge_colors)}
        for c, e in zip(col_in.tolist(), e_in.tolist()):
            infl[c] = np.array([e * N + N - 1, 1], dtype=np.int32)
        for c, e in zip(col_out.tolist(), e_out.tolist()):
            outfl[c] = np.array([e * N, 0], dtype=np.int32)
        return infl, outfl
    for c in range(network_mesh.num_edge_colors):
        ei = e_in[colors[e_in] == c]
        eo = e_out[colors[e_out] == c]
        infl[c] = np.stack([ei * N + N - 1, np.ones_like(ei)], axis=1).astype(np.int32).ravel()
        outfl[c] = np.stack([eo * N, np.zeros_like(eo)], axis=1).astype(np.int32).ravel()
    return infl, outfl


def _is_cuda_tensor(v) -> bool:
    torch = sys.modules.get("torch")  # a tensor exists only once torch has been imported
    return torch is not None and isinstance(v, torch.Tensor) and v.is_cuda


def _check_cuda_tensor(t, dev, name: str) -> None:
    """Device inputs are taken as they are: float64, contiguous, on the mesh's GPU."""
    import torch  # noqa: PLC0415

    if t.dtype != torch.float64:
        raise TypeError(f"{name}: CUDA tensors must be float64, got {t.dtype} (no implicit conversion)")
    if t.device.index != dev.index:
        raise ValueError(f"{name} is on {t.device}, the mesh on cuda:{dev.index}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous tensor")


class BlockForm:
    """Placeholder for a compiled DOLFINx form: records which block of the system it is."""

    def __init__(self, kind: str, test: int, trial: int | None = None):
        self.kind = kind
        self.test = test
        self.trial = trial
        self.rank = 1 if trial is None else 2

    def __repr__(self):
        return f"BlockForm({self.kind!r}, test={self.test}, trial={self.trial})"


class HydraulicNetworkAssembler:
    """Assembler for the variational formulation of a hydraulic network (assembly.py:95-162).

    Args:
        mesh: The network mesh
        flux_degree: polynomial degree of the flux (1 supported on the GPU path)
        pressure_degree: polynomial degree of the pressure (0 supported on the GPU path)
    """

    @timed("nxfx:HydraulicNetworkAssembler:__init__")
    def __init__(self, mesh: NetworkMesh, flux_degree: int = 1, pressure_degree: int = 0):
        flux_degree, pressure_degree = int(flux_degree), int(pressure_degree)
        if flux_degree < 1 or pressure_degree < 0 or flux_degree > 4 or pressure_degree > 3:
            raise ValueError("flux_degree in 1..4 and pressure_degree in 0..3 are supported")
        self._network_mesh = mesh
        self._degrees = (flux_degree, pressure_degree)
        # (1, 0) -- the reference's defaults, used by every demo -- runs on the specialised kernels;
        # other degrees use the table-driven path (generic.py / generic.cuh)
        self._generic = None
        if self._degrees != (1, 0):
            from .generic import build_generic_system  # noqa: PLC0415

            self._generic = build_generic_system(mesh, flux_degree, pressure_degree)
        N = mesh.cells_per_edge
        E = mesh.graph_edges.shape[0]
        C_ = mesh.num_edge_colors
        counts = mesh._color_count
        per_edge = flux_degree * N + 1
        qoff = np.concatenate([[0], np.cumsum(counts * per_edge)])
        self._flux_spaces = _FluxSpaces(mesh, qoff, flux_degree)
        nv = mesh.mesh.topology.index_map(0).size_local
        n_p = N * E if pressure_degree == 0 else nv + (pressure_degree - 1) * N * E
        if pressure_degree == 0:
            pdofs = lambda: np.arange(N * E, dtype=np.int32)[:, None]  # noqa: E731
        else:
            pdofs = lambda: (self._generic.cell_pressure_dofs - int(qoff[-1])).astype(np.int32)  # noqa: E731
        self._pressure_space = FunctionSpace(
            mesh.mesh, pressure_degree, pressure_degree == 0, n_p, int(qoff[-1]), pdofs, "pressure",
        )
        n_bif = mesh.bifurcation_values.size
        self._lm_space = FunctionSpace(
            mesh.lm_mesh, 0, True, n_bif, int(qoff[-1]) + n_p,
            lambda: np.arange(n_bif, dtype=np.int32)[:, None], "lm",
        )
        self._block_sizes = [int(c) * per_edge for c in counts] + [n_p, n_bif]
        self._n_dofs = int(sum(self._block_sizes))
        # integration data (assembly.py:152-162)
        self._integration_data = []
        self._in_idx = max(mesh.in_marker, mesh.out_marker) + 1
        in_flux_entities, out_flux_entities = compute_integration_data(mesh)
        self._in_keys = tuple(in_flux_entities.keys())
        self._out_keys = tuple(out_flux_entities.keys())
        for color in self._in_keys:
            self._integration_data.append((self._in_idx + color, in_flux_entities[color]))
        self._out_idx = self._in_idx + len(out_flux_entities)
        for color in self._out_keys:
            self._integration_data.append((self._out_idx + color, out_flux_entities[color]))
        self._a = None
        self._L = None
        self._pbc_d = None
        self._R = (None, 1.0)
        self._f = (None, 0.0)
        self._symbolic_done = False

    # ---- forms --------------------------------------------------------------------------------
    @timed("nxfx:HydraulicNetworkAssembler:compute_forms")
    def compute_forms(
        self,
        p_bc_ex,
        f=None,
        R=None,
        jit_options: dict | None = None,
        form_compiler_options: dict | None = None,
    ):
        """Set the data of the weak form (assembly.py:164-299).

        Args:
            p_bc_ex: boundary pressure: callable ``p(x)`` with ``x`` of shape (3, npoints)
                (DOLFINx interpolation convention), a :class:`fem.CoordinateExpr`
                (``SpatialCoordinate(mesh)[i]`` arithmetic), an object with ``eval(x)``, or an array
                of vertex values (NumPy, or a CUDA ``torch.Tensor``).
            f: source term: ``None`` (0), a float, or an array with one value per cell.
            R: resistance: ``None`` (1), a float, an array per cell or per graph edge.
            jit_options, form_compiler_options: accepted for signature compatibility; there is no
                JIT (the element kernels are compiled ahead of time into libnxfx_b200).

        Arrays may be CUDA tensors (``torch.Tensor``): float64, contiguous, one-dimensional, on the mesh's device
        (anything else raises before any work is enqueued; nothing is converted).  They are read as the
        NumPy arrays are, at this call: the assembler copies them into its own device buffers on the
        library's stream, after the work the current torch stream has enqueued so far (an event, no host
        wait), and the caller may free or overwrite them as soon as the call returns.  With device inputs
        only, the call does not wait for the device.  On a partitioned network ``R`` / ``f`` tensors of the
        whole network's size are restricted to this rank's edges on the device (``nxfx_gather``).
        """
        nm = self._network_mesh
        dev = nm.device
        nv = nm.mesh.topology.index_map(0).size_local
        nc = nm.mesh.topology.index_map(1).size_local
        # CUDA tensors: every check before anything is enqueued
        pbc_t = p_bc_ex if _is_cuda_tensor(p_bc_ex) else None
        if pbc_t is not None:
            _check_cuda_tensor(pbc_t, dev, "p_bc")
            if tuple(pbc_t.shape) != (nv,):
                raise ValueError(f"p_bc array must have one value per mesh vertex ({nv})")
        R_plan = self._device_coef_plan(R, nc, "R")
        f_plan = self._device_coef_plan(f, nc, "f")
        tensors = [t for t in (pbc_t, R if R_plan else None, f if f_plan else None) if t is not None]
        if tensors:
            dev.wait_for_torch(*tensors)
        # p_bc interpolated into P1 on the parent mesh (assembly.py:225-234)
        if pbc_t is not None:
            self._set_pbc_device(pbc_t, nv)
        elif isinstance(p_bc_ex, np.ndarray):
            pbc = np.ascontiguousarray(p_bc_ex, dtype=np.float64)
            if pbc.shape != (nv,):
                raise ValueError(f"p_bc array must have one value per mesh vertex ({nv})")
        else:
            fn = p_bc_ex.eval if hasattr(p_bc_ex, "eval") and not callable(p_bc_ex) else p_bc_ex
            if not callable(fn):
                raise TypeError(
                    "p_bc_ex must be a callable p(x), a fem.CoordinateExpr, or an array of vertex "
                    "values (UFL expressions need UFL/FFCx, which this build does not use)"
                )
            x = nm.mesh.geometry.x
            pbc = np.ascontiguousarray(np.asarray(fn(x.T), dtype=np.float64) * np.ones(nv))
        if pbc_t is None:
            self._pbc_host = pbc
            self._ensure_pbc_buffer(nv)
            # the forms read p_bc at BOUNDARY vertices only (assembly.py:258-260): when those are a few contiguous
            # runs of vertex ids (generated trees: the inlet and the last generation) only the runs travel over PCIe
            runs = self._boundary_runs()
            if runs is None:
                self._pbc_d.upload(pbc, sync=False)
                self.pbc_h2d_bytes = pbc.nbytes
            else:
                for a, b in runs:
                    dev.call("nxfx_memcpy_h2d", C.c_void_p(self._pbc_d.ptr + 8 * a), C.c_void_p(pbc.ctypes.data + 8 * a),
                             C.c_size_t(8 * (b - a)))
                self.pbc_h2d_bytes = int(sum(8 * (b - a) for a, b in runs))
            dev.call("nxfx_set_boundary_pressure", self._pbc_d.c_ptr)  # into the vertex records
            dev.sync()
        nm._pbc_owner = self  # the vertex records now hold THIS assembler's boundary data
        if R_plan:
            self._R = self._gather_coef(R, R_plan, nc, self._R[0])
        else:
            self._R = self._coefficient(R, 1.0, nc, "R", self._R[0])
        if f_plan:
            self._f = self._gather_coef(f, f_plan, nc, self._f[0])
        else:
            self._f = self._coefficient(f, 0.0, nc, "f", self._f[0])
        C_ = nm.num_edge_colors
        self._a = _BilinearBlocks(C_)
        self._L = _LinearBlocks(C_)

    def _ensure_pbc_buffer(self, nv: int) -> None:
        if self._pbc_d is None or self._pbc_d.n != nv:
            self._pbc_d = self._network_mesh.device.empty(nv)
            self._pbc_d.zero()

    def _set_pbc_device(self, pbc_t, nv: int) -> None:
        """p_bc from a checked CUDA tensor: device-to-device into the assembler's own copy (the boundary runs only
        when :meth:`_boundary_runs` finds them), then into the vertex records; no host wait."""
        dev = self._network_mesh.device
        self._pbc_host = None
        self._ensure_pbc_buffer(nv)
        src = pbc_t.data_ptr()
        runs = self._boundary_runs()
        for a, b in [(0, nv)] if runs is None else runs:
            if b > a:
                dev.call("nxfx_memcpy_d2d", C.c_void_p(self._pbc_d.ptr + 8 * a), C.c_void_p(src + 8 * a),
                         C.c_size_t(8 * (b - a)))
        self.pbc_h2d_bytes = 0
        dev.call("nxfx_set_boundary_pressure", self._pbc_d.c_ptr)

    def _device_coef_plan(self, val, nc: int, name: str):
        """``(rows, S)`` of the ``nxfx_gather`` that turns a CUDA tensor coefficient into one value per cell
        (``rows``: ``"local"`` or ``"global"`` -- a whole-network array on a partitioned mesh), ``None`` for
        anything that is not a CUDA tensor.  Checks the tensor; the sizes are tried in the order of
        :meth:`_coefficient`."""
        if not _is_cuda_tensor(val):
            return None
        nm = self._network_mesh
        _check_cuda_tensor(val, nm.device, name)
        N, E = nm.cells_per_edge, nm.graph_edges.shape[0]
        n = val.numel() if val.dim() == 1 else -1
        if getattr(nm, "_partition", None) is not None and n >= 0 and n != nc:
            Eg = nm._global_graph.number_of_edges()
            if n == Eg:
                return ("global", 1)
            if n == Eg * N:
                return ("global", N)
        if n == E:
            return ("local", 1)
        if n == nc:
            return ("local", N)
        raise ValueError(f"{name} must be a scalar, one value per cell ({nc}) or per graph edge")

    def _gather_coef(self, t, plan, nc: int, previous=None):
        """Per-cell device copy of a checked CUDA tensor coefficient (``previous`` reused when it has the size)."""
        nm = self._network_mesh
        dev = nm.device
        rows, S = plan
        out = previous if previous is not None and previous.n == nc else dev.empty(nc)
        gmap = None
        if rows == "global":
            if getattr(nm, "_global_edges_d", None) is None:  # uploaded once per mesh
                nm._global_edges_d = dev.from_host(np.ascontiguousarray(nm._partition.global_edges, dtype=np.int32))
            gmap = nm._global_edges_d.c_ptr
        dev.call("nxfx_gather", C.c_void_p(t.data_ptr()), gmap, S, nm.graph_edges.shape[0], nm.cells_per_edge,
                 out.c_ptr)
        return (out, 0.0)

    def _boundary_runs(self, max_runs: int = 8):
        """``[(first, last + 1), ...]`` of the boundary vertex ids if they form at most ``max_runs`` contiguous
        runs, else ``None`` (upload everything)."""
        if not hasattr(self, "_pbc_runs"):
            bv = np.sort(np.asarray(self._network_mesh.boundary_values, dtype=np.int64))
            runs = None
            if bv.size:
                cut = np.flatnonzero(np.diff(bv) != 1)
                if cut.size + 1 <= max_runs:
                    starts = np.concatenate([[0], cut + 1])
                    ends = np.concatenate([cut, [bv.size - 1]])
                    runs = [(int(bv[a]), int(bv[b]) + 1) for a, b in zip(starts, ends)]
            self._pbc_runs = runs
        return self._pbc_runs

    def _coefficient(self, val, default, nc, name, previous=None):
        """``previous``: the device array of the last call -- reused (no allocation, asynchronous upload)
        when the new coefficient is an array of the same size, e.g. in a time loop."""
        if val is None:
            return (None, float(default))
        if np.isscalar(val) or (hasattr(val, "value") and np.ndim(val.value) == 0):
            return (None, float(getattr(val, "value", val)))
        arr = np.asarray(val, dtype=np.float64)
        nm = self._network_mesh
        part = getattr(nm, "_partition", None)
        if part is not None and arr.ndim == 1 and arr.size != nc:
            # partitioned network: coefficients given for the GLOBAL network are restricted to this rank's edges
            Eg, Nc = nm._global_graph.number_of_edges(), nm.cells_per_edge
            if arr.size == Eg:
                arr = arr[part.global_edges]
            elif arr.size == Eg * Nc:
                arr = arr.reshape(Eg, Nc)[part.global_edges].ravel()
        if arr.shape == (nm.graph_edges.shape[0],) and nm.cells_per_edge != 1:
            arr = np.repeat(arr, nm.cells_per_edge)
        if arr.shape != (nc,):
            raise ValueError(f"{name} must be a scalar, one value per cell ({nc}) or per graph edge")
        arr = np.ascontiguousarray(arr)
        if previous is not None and previous.n == arr.size:
            previous.upload(arr, sync=False)  # ordered on the context's stream before the next assembly
            self._coef_keepalive = getattr(self, "_coef_keepalive", {})
            self._coef_keepalive[name] = arr  # the asynchronous copy reads the host array
            return (previous, 0.0)
        return (nm.device.from_host(arr), 0.0)

    # ---- accessors (assembly.py:301-326, 370-398) -------------------------------------------------
    @property
    def lm_space(self) -> FunctionSpace:
        """The function space of the bifurcation Lagrange multipliers"""
        return self._lm_space

    @property
    def pressure_space(self) -> FunctionSpace:
        return self._pressure_space

    @property
    def flux_spaces(self):
        """Function spaces of the flux, one per edge colour."""
        return self._flux_spaces

    @property
    def function_spaces(self):
        """All spaces in the order ``[flux, pressure, lm]`` used by :py:meth:`assemble`."""
        return [*self._flux_spaces, self._pressure_space, self._lm_space]

    @property
    def network(self) -> NetworkMesh:
        return self._network_mesh

    @property
    def block_sizes(self) -> list[int]:
        return self._block_sizes

    @property
    def degrees(self) -> tuple[int, int]:
        """(flux_degree, pressure_degree)"""
        return self._degrees

    @property
    def is_generic(self) -> bool:
        """True when the table-driven higher-order path is used."""
        return self._generic is not None

    @property
    def num_dofs(self) -> int:
        return self._n_dofs

    @property
    def bilinear_forms(self):
        if self._a is None:
            logging.error("Bilinear forms haven't been computed. Need to call compute_forms()")
        else:
            return self._a

    def bilinear_form(self, i: int, j: int):
        a = self.bilinear_forms
        if i > len(a) or j > len(a[i]):
            logging.error("Bilinear form a[" + str(i) + "][" + str(j) + "] out of range")
        return a[i][j]

    @property
    def linear_forms(self):
        if self._L is None:
            logging.error("Linear forms haven't been computed. Need to call compute_forms()")
        else:
            return self._L

    def linear_form(self, i: int):
        L = self.linear_forms
        if i > len(L):
            logging.error("Linear form L[" + str(i) + "] out of range")
        return L[i]

    # ---- matrices / vectors ------------------------------------------------------------------------
    def create_matrix(self, kind=None) -> Mat:
        """Symbolic phase (``fem.petsc.create_matrix``, solver.py:43 / assembly.py:354): builds the
        CSR pattern on the device."""
        if self._a is None:
            raise RuntimeError("compute_forms() must be called before creating the matrix")
        dev = self._network_mesh.device
        nm = self._network_mesh
        owner = getattr(nm, "_pattern_degrees", None)
        if owner is not None and owner != self._degrees:
            # one sparsity pattern per device context: a second assembler with other degrees would
            # silently replace the pattern under the first one's matrices
            raise RuntimeError(
                f"this NetworkMesh already carries the pattern of a flux/pressure degree {owner} assembler; "
                f"build a second NetworkMesh for degrees {self._degrees}"
            )
        if not self._symbolic_done and owner is not None:
            self._symbolic_done = True  # same degrees: the pattern on the device is the one we need
        if not self._symbolic_done:
            nm._pattern_degrees = self._degrees
            if self._generic is None:
                dev.call("nxfx_symbolic")
            else:
                from . import _lib  # noqa: PLC0415

                g = self._generic
                c32 = lambda a: _lib.as_i32p(np.ascontiguousarray(a, dtype=np.int32))  # noqa: E731
                c64 = lambda a: _lib.as_f64p(np.ascontiguousarray(a, dtype=np.float64))  # noqa: E731
                dev.call(
                    "nxfx_set_generic_system", g.n_dofs, g.n_flux, g.colidx.size, c32(g.rowptr), c32(g.colidx),
                    c32(g.src_id), c64(g.src_coef), c32(g.bsrc_ptr), c32(g.bsrc_id), c64(g.bsrc_coef),
                )
                dev.sync()
                # analysis phase of the direct solve for these degrees (condense.py / condense.cuh)
                from .condense import build_condensation  # noqa: PLC0415

                cd = build_condensation(nm, *self._degrees)
                t = cd.packed()
                dev.call(
                    "nxfx_set_condensation", int(cd.pd >= 1), cd.fd * cd.N + 1, cd.n_max, cd.kl, cd.pcell_base,
                    cd.pcell_stride, c32(t["type_n"]), c32(t["loc_ptr"]), c32(t["loc_kind"]), c32(t["loc_off"]),
                    c32(t["k_ptr"]), c32(t["k_row"]), c32(t["k_col"]), c32(t["k_cell"]), c64(t["k_coef"]),
                    c32(t["c_ptr"]), c32(t["c_row"]), c32(t["c_slot"]), c64(t["c_coef"]),
                    c32(t["d_ptr"]), c32(t["d_slot"]), c32(t["d_col"]), c64(t["d_coef"]), c32(cd.bif_node),
                )
            self._symbolic_done = True
        nnz = C.c_int64()
        dev.call("nxfx_get_sizes", None, None, None, C.byref(nnz))
        return Mat(dev, self._n_dofs, nnz.value, self._block_sizes, kind="nest" if kind == "nest" else kind)

    def create_vector(self, kind=None) -> Vec:
        return Vec(self._network_mesh.device, self._n_dofs, self._block_sizes, kind=kind)

    @timed("nxfx:HydraulicNetworkAssembler:assemble")
    def assemble(
        self,
        A: Mat | None = None,
        b: Vec | None = None,
        assemble_lhs: bool = True,
        assemble_rhs: bool = True,
        kind=None,
    ) -> tuple[Mat, Vec]:
        """Assemble system matrix and rhs vector (assembly.py:328-368).

        If ``A``/``b`` are given the contributions are ADDED to them (PETSc ``ADD_VALUES``) unless
        they were zeroed (``zeroEntries``), in which case the kernel overwrites without reading.
        """
        if self._a is None:
            raise RuntimeError("compute_forms() must be called before assemble()")
        dev = self._network_mesh.device
        if assemble_lhs and A is None:
            A = self.create_matrix(kind=kind)
        if assemble_lhs:
            kind = "nest" if A.getType() == "nest" else kind
        if assemble_rhs and b is None:
            b = self.create_vector(kind=kind)
            b.zeroEntries()
        nm = self._network_mesh
        if getattr(nm, "_pbc_owner", None) is not self and assemble_rhs:
            # another assembler on the same network set its boundary data since: restore ours
            dev.call("nxfx_set_boundary_pressure", self._pbc_d.c_ptr)
            nm._pbc_owner = self
        if assemble_lhs:
            A.bind()
        # zeroed targets are overwritten without being read; otherwise ADD_VALUES semantics
        a_zero = A.consume_zero() if assemble_lhs else True
        b_zero = (b._zero_pending and not b._host_dirty) if assemble_rhs else True
        if assemble_lhs and assemble_rhs and a_zero != b_zero:
            if a_zero:
                A.zero_now()
            acc = True
        else:
            acc = not (a_zero if assemble_lhs else b_zero)
        b_ptr = None
        if assemble_rhs:
            b_ptr = b.device_ptr() if acc else b.device_ptr_overwrite()
        R_d, R_c = self._R
        f_d, f_c = self._f
        dev.call(
            "nxfx_assemble" if self._generic is None else "nxfx_assemble_generic",
            R_d.c_ptr if R_d is not None else None, C.c_double(R_c),
            f_d.c_ptr if f_d is not None else None, C.c_double(f_c),
            int(bool(assemble_lhs)), int(bool(assemble_rhs)), int(acc), b_ptr,
        )
        if assemble_lhs:
            A.assembled = True
        if assemble_rhs:
            b.mark_device_modified()
        return (A, b)


class _FluxSpaces:
    """Sequence of the per-colour flux spaces, built on demand (``C == E`` in uncoloured mode)."""

    def __init__(self, mesh: NetworkMesh, qoff, degree):
        self._mesh, self._qoff, self._degree = mesh, qoff, degree
        self._cache: dict[int, FunctionSpace] = {}

    def __len__(self):
        return self._mesh.num_edge_colors

    def __getitem__(self, c):
        if isinstance(c, slice):
            return [self[i] for i in range(*c.indices(len(self)))]
        if c < 0:
            c += len(self)
        if not 0 <= c < len(self):
            raise IndexError(c)
        if c not in self._cache:
            N = self._mesh.cells_per_edge
            n_edges = int(self._mesh._color_count[c])
            fd = self._degree
            per_edge = fd * N + 1

            def cell_dofs(n_edges=n_edges, N=N, fd=fd, per_edge=per_edge):
                eb = np.repeat(np.arange(n_edges) * per_edge, N)
                j = np.tile(np.arange(N), n_edges)
                cols = [eb + j, eb + j + 1] + [eb + (N + 1) + j * (fd - 1) + i for i in range(fd - 1)]
                return np.stack(cols, axis=1)

            self._cache[c] = FunctionSpace(
                self._mesh.submeshes[c], fd, False, n_edges * per_edge, int(self._qoff[c]),
                cell_dofs, f"flux_{c}",
            )
        return self._cache[c]

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class _BilinearBlocks:
    """``(C+2) x (C+2)`` nested list of forms with ``None`` for empty blocks (assembly.py:284-299):
    ``a[i][i]`` mass, ``a[P][i]`` / ``a[i][P]`` pressure coupling, ``a[LM][i]`` / ``a[i][LM]``
    multiplier coupling."""

    def __init__(self, C_: int):
        self._C = C_

    def __len__(self):
        return self._C + 2

    def __getitem__(self, i):
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        return _BilinearRow(self._C, i)

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class _BilinearRow:
    def __init__(self, C_: int, i: int):
        self._C, self._i = C_, i

    def __len__(self):
        return self._C + 2

    def __getitem__(self, j):
        C_, i = self._C, self._i
        if j < 0:
            j += len(self)
        if not 0 <= j < len(self):
            raise IndexError(j)
        P, LM = C_, C_ + 1
        if i < C_:
            if j == i:
                return BlockForm("mass", i, j)
            if j == P:
                return BlockForm("minus_grad_T", i, j)
            if j == LM:
                return BlockForm("multiplier_T", i, j)
            return None
        if j < C_:
            return BlockForm("grad" if i == P else "multiplier", i, j)
        return None

    def __iter__(self):
        return (self[j] for j in range(len(self)))


class _LinearBlocks:
    def __init__(self, C_: int):
        self._C = C_

    def __len__(self):
        return self._C + 2

    def __getitem__(self, i):
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        kind = "boundary_pressure" if i < self._C else ("source" if i == self._C else "zero")
        return BlockForm(kind, i)

    def __iter__(self):
        return (self[i] for i in range(len(self)))
