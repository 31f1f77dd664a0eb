"""Solver interface for network problems (drop-in for ``networks_fenicsx.solver.Solver``,
solver.py:16-143).  PETSc KSP / MUMPS are replaced by the device solver behind ``nxfx_solve``:
the network Schur-complement preconditioner (exact on tree networks, for every polynomial degree)
used either as a direct solver with iterative refinement (``ksp_type=preonly``, the reference's default with
``pc_type=lu``) or inside flexible GMRES."""

from __future__ import annotations

import ctypes as C
import typing

import numpy as np

from . import _lib, assembly
from .common import timed
from .fem import Function
from .la import KSP, Mat, Vec
from .schedule import build_tree_schedule

__all__ = ["Solver"]

_DIRECT_PCS = {"lu", "cholesky", "schur", "network_schur", "fieldsplit"}


class Solver:
    """Solver interface for the network problems.

    Args:
        assembler: The hydraulic network assembler.
        petsc_options_prefix: Prefix for the options (kept for compatibility).
        petsc_options: Dictionary of PETSc-style options, see :class:`la.KSP`. Extra keys:
            ``nxfx_refine_steps`` (iterative-refinement steps of the direct solve, default 1),
            ``nxfx_final_residual`` (also evaluate the true residual of the final iterate),
            ``nxfx_refine_rtol`` (default 1e-13: refinement stops as soon as the iterate has that relative
            residual; 0 = always apply ``nxfx_refine_steps`` corrections).
        kind: ``None``/``"mpi"`` (monolithic AIJ) or ``"nest"``.
    """

    def __init__(
        self,
        assembler: assembly.HydraulicNetworkAssembler,
        petsc_options_prefix: str = "NetworkSolver_",
        petsc_options: dict | None = None,
        kind: str | typing.Sequence[typing.Sequence[str]] | None = None,
        schedule=None,
    ):
        self._assembler = assembler
        nm = assembler.network
        self._ksp = KSP(nm.comm)
        # symbolic phase (solver.py:43-49)
        if kind is not None and not isinstance(kind, str):
            # a list of lists of PETSc matrix types (solver.py:37, fem.petsc.create_matrix): a MatNest whose
            # blocks have the given types.  Storage here is one CSR with block views either way.
            rows = [list(r) for r in kind]
            nb = len(assembler.block_sizes)
            if len(rows) != nb or any(len(r) != nb for r in rows):
                raise ValueError(f"kind as a list of lists must be {nb} x {nb} (blocks [flux colours, pressure, lm])")
            kind = "nest"
        self._A = assembler.create_matrix(kind=kind)
        kind = "nest" if self._A.getType() == "nest" else kind
        self._b = assembler.create_vector(kind=kind)
        self._x = assembler.create_vector(kind=kind)
        self.ksp.setOperators(self.A)
        self.ksp.setOptionsPrefix(petsc_options_prefix)
        self._A.setOptionsPrefix(f"{petsc_options_prefix}A_")
        self._b.setOptionsPrefix(f"{petsc_options_prefix}b_")
        if petsc_options is None:
            petsc_options = {
                "ksp_type": "preonly",
                "pc_type": "lu",
                "pc_factor_mat_solver_type": "mumps",
                "ksp_monitor": None,
                "ksp_error_if_not_converged": True,
            }
        self.ksp.options = dict(petsc_options)
        # elimination schedule of the bifurcation graph (the analysis phase of the direct solver)
        # (``schedule``: a precomputed one, e.g. the local part of a partitioned network)
        if schedule is None and getattr(nm, "_partition", None) is not None:
            schedule = nm._partition.schedule  # this rank's chunks + the replicated top chunk
        self._schedule = schedule if schedule is not None else build_tree_schedule(
            nm.graph_edges, nm.node_multiplier_index, nm.bifurcation_values.size,
            root_hint_nodes=nm._boundary_out_nodes,
        )
        s = self._schedule
        nm.device.call(
            "nxfx_set_tree_schedule",
            _lib.as_i32p(s.t_of_bif), _lib.as_i32p(s.t_parent), _lib.as_i32p(s.t_pedge),
            _lib.as_i32p(s.t_cptr), _lib.as_i32p(s.t_cidx), s.n_chunks, _lib.as_i32p(s.chunk_lptr),
            s.lvl_ptr.size, _lib.as_i32p(s.lvl_ptr), s.chord_edge.size, _lib.as_i32p(s.chord_edge),
        )
        self.info = _lib.SolveInfo()
        self._x_stage = None
        # partitioned network (NetworkMesh under torchrun): the solve goes through the distributed layer
        self._dist = None
        if getattr(nm, "_partition", None) is not None and not getattr(self, "_no_dist", False):
            from .distributed import DistributedSolver  # noqa: PLC0415

            self._dist = DistributedSolver.from_solver(self, nm._partition)

    @property
    def assembler(self) -> assembly.HydraulicNetworkAssembler:
        """The hydraulic network assembler."""
        return self._assembler

    @property
    def A(self) -> Mat:
        """System matrix."""
        return self._A

    @property
    def b(self) -> Vec:
        """Right-hand side vector."""
        return self._b

    @property
    def x(self) -> Vec:
        """Solution vector (blocked ``[flux colours, pressure, multipliers]``)."""
        return self._x

    @property
    def ksp(self) -> KSP:
        return self._ksp

    def create_functions(self) -> list[Function]:
        """Functions ``[flux_color_i ..., pressure, global_flux]`` backed by pinned host memory; pass
        them to :meth:`solve` to have the solution copied straight into them (no staging copy)."""
        asm = self.assembler
        dev = asm.network.device
        out = []
        spaces = [*asm.flux_spaces, asm.pressure_space, asm.lm_space]
        names = [f"flux_color_{i}" for i in range(len(spaces) - 2)] + ["pressure", "global_flux"]
        # ONE pinned buffer in block order, the functions are views into it: solve() has the library mirror x into
        # it while the residual check still runs (nxfx_set_solution_mirror)
        mirror = dev.pinned(asm.num_dofs)
        off = 0
        for V, name in zip(spaces, names):
            fn = Function(V, name=name, array=mirror[off:off + V.num_dofs])
            fn._pinned = True
            fn._mirror = mirror
            off += V.num_dofs
            out.append(fn)
        return out

    def assemble(self, lhs: bool = True, rhs: bool = True):
        """Zero and re-assemble the system matrix and rhs vector (solver.py:90-101)."""
        if self._A is not None and lhs:
            self._A.zeroEntries()
        if self._b is not None and rhs:
            self._b.zeroEntries()
        self.assembler.assemble(self._A, self._b, assemble_lhs=lhs, assemble_rhs=rhs)

    # ---- options ------------------------------------------------------------------------------
    def solve_options(self) -> _lib.SolveOpts:
        o = self.ksp.options
        ksp_type = str(o.get("ksp_type", "preonly")).lower()
        pc_type = str(o.get("pc_type", "lu")).lower()
        opts = _lib.SolveOpts()
        # (higher-order elements take the same route: their exact condensation -- per-edge banded LU + 2 x 2 node
        # blocks over the same schedule, condense.py / condense.cuh -- sits behind PC_NETWORK_SCHUR too)
        if pc_type in _DIRECT_PCS:
            opts.pc_type = _lib.PC_NETWORK_SCHUR
        elif pc_type == "none":
            opts.pc_type = _lib.PC_NONE
        elif pc_type == "jacobi":
            opts.pc_type = _lib.PC_JACOBI_FLUX
        else:
            raise ValueError(f"unsupported pc_type {pc_type!r}")
        direct = opts.pc_type == _lib.PC_NETWORK_SCHUR
        if ksp_type == "preonly":
            # on graphs with cycles the Schur preconditioner is a spanning-tree approximation:
            # direct-solver accuracy then needs the Krylov wrapper
            opts.ksp_type = _lib.KSP_PREONLY if (self._schedule.is_forest or not direct) else _lib.KSP_FGMRES
        elif ksp_type in ("gmres", "fgmres", "minres", "cg", "bcgs", "richardson"):
            opts.ksp_type = _lib.KSP_FGMRES
        else:
            raise ValueError(f"unsupported ksp_type {ksp_type!r}")
        # preonly: the checked residual is the one BEFORE the last refinement correction
        default_rtol = 1e-10 if ksp_type == "preonly" else 1e-5  # 1e-5: PETSc default for Krylov types
        opts.rtol = float(o.get("ksp_rtol", default_rtol))
        opts.atol = float(o.get("ksp_atol", 1e-50 if ksp_type != "preonly" else 1e-300))
        opts.max_it = int(o.get("ksp_max_it", 10000))
        opts.restart = int(o.get("ksp_gmres_restart", 30))
        opts.refine_steps = int(o.get("nxfx_refine_steps", 1))
        opts.error_if_not_converged = int(bool(o.get("ksp_error_if_not_converged", False)))
        opts.final_residual = int(bool(o.get("nxfx_final_residual", False)))
        opts.refine_rtol = float(o.get("nxfx_refine_rtol", 1e-13))
        return opts

    # ---- solve --------------------------------------------------------------------------------
    @timed("nxfx:Solver:solve")
    def solve(self, functions: list[Function] | None = None) -> list[Function]:
        """Solve the linear system and assign the blocks of the solution to functions named
        ``flux_color_i``, ``pressure`` and ``global_flux`` (the multipliers), solver.py:107-135.

        Args:
            functions: functions to assign to (reused across solves to avoid host allocations);
                created from the assembler's spaces if not given.
        """
        asm = self.assembler
        dev = asm.network.device
        if functions is None:
            # fresh Functions per call (as the reference does); their arrays are filled from a
            # pinned staging buffer that the solver keeps, so repeated solves do not pay for
            # page-locking 8*n_dofs bytes every time
            functions = []
            for i, Vi in enumerate(asm.flux_spaces):
                functions.append(Function(Vi, name=f"flux_color_{i}", array=np.empty(Vi.num_dofs)))
            functions.append(Function(asm.pressure_space, name="pressure", array=np.empty(asm.pressure_space.num_dofs)))
            functions.append(Function(asm.lm_space, name="global_flux", array=np.empty(asm.lm_space.num_dofs)))
            staged = True
        else:
            staged = not all(getattr(fn, "_pinned", False) for fn in functions)
        opts = self.solve_options()
        self.info = _lib.SolveInfo()
        self._A._materialise_zero()
        self._A.bind()
        mirror = getattr(functions[0], "_mirror", None) if not staged else None
        if mirror is not None and not all(getattr(fn, "_mirror", None) is mirror for fn in functions):
            mirror = None
        # the library fills the mirror itself wherever the solve goes through nxfx_solve
        mirrored = mirror is not None and (self._dist is None or self._dist.exchange == "peer")
        if mirrored:
            dev.call("nxfx_set_solution_mirror", C.c_void_p(mirror.ctypes.data))
        try:
            self._run_solve(opts, dev)
        finally:
            if mirrored:
                dev.call("nxfx_set_solution_mirror", None)
        self._x.mark_device_modified()
        # fem.petsc.assign: split the blocked vector into the functions (solver.py:134)
        if sum(fn.x.array.size for fn in functions) != self._x.n:
            raise ValueError("functions do not match the block layout [flux colours, pressure, multipliers]")
        if staged:
            if self._x_stage is None:
                self._x_stage = dev.pinned(self._x.n)
            self._x.d.download(self._x_stage)  # one D2H, synchronises
            off = 0
            for fn in functions:
                n = fn.x.array.size
                np.copyto(fn.x.array, self._x_stage[off:off + n])
                off += n
        elif mirrored:  # Solver.create_functions(): the library has already mirrored x into the views
            pass
        elif mirror is not None:
            self._x.d.download(mirror)  # one D2H into the buffer behind the views, synchronises
        else:  # caller-provided pinned arrays: D2H straight into them
            off = 0
            for fn in functions:
                n = fn.x.array.size
                if n:
                    dev.call(
                        "nxfx_memcpy_d2h", C.c_void_p(fn.x.array.ctypes.data),
                        C.c_void_p(self._x.d.ptr + 8 * off), C.c_size_t(8 * n),
                    )
                off += n
            dev.sync()
        return functions

    def _run_solve(self, opts, dev) -> None:
        if self._dist is not None:
            hist = self._dist.solve(refine_steps=int(opts.refine_steps), final_residual=bool(opts.final_residual),
                                    refine_rtol=float(opts.refine_rtol))
            self.ksp.its = 1 + self._dist.corrections
            self.ksp.history = [h * self._dist.rhs_norm for h in hist]
            self.ksp.rnorm = self.ksp.history[-1] if hist else float("nan")
            converged = bool(hist) and hist[-1] <= max(opts.rtol, 0.0) or not hist
            self.ksp.reason = 2 if converged else -3
            if not converged and opts.error_if_not_converged:
                raise RuntimeError(f"nxfx_solve failed (-3): linear solve did not converge: relative residual {hist[-1]:.3e}")
        else:
            try:
                dev.call(
                    "nxfx_solve", self._b.device_ptr(), self._x.device_ptr_overwrite(),
                    C.byref(opts), C.byref(self.info),
                )
            finally:
                self._record_info()

    def _record_info(self):
        info = self.info
        self.ksp.its = int(info.iterations)
        self.ksp.rnorm = float(info.residual_norm)
        self.ksp.reason = 2 if info.converged else -3
        self.ksp.history = [info.history[i] for i in range(info.history_len)]
        if "ksp_monitor" in self.ksp.options and self.ksp.options.get("nxfx_print_monitor", False):
            for i, r in enumerate(self.ksp.history):
                print(f"  {i} KSP Residual norm {r:.12e}")

    def __del__(self):
        return None
