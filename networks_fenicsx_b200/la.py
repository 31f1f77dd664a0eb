"""PETSc ``Vec`` / ``Mat`` / ``KSP`` stand-ins backed by device memory (petsc4py is not available
on the GPU boxes).  They answer the calls the reference and its users make on the objects returned
by ``assemble()`` / ``Solver`` (solver.py:43-56,97-101,127-134; assembly.py:352-367):
``getSize, getType, zeroEntries, assemble, mult, getValuesCSR, getNestSubMatrix, norm, array, ...``.
If petsc4py is importable, ``Mat.to_petsc()`` / ``Vec.to_petsc()`` hand over real PETSc objects.
"""

from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from .device import Device, DeviceArray


class Vec:
    """Blocked vector ``[q_0 .. q_{C-1}, p, lambda]`` (assembly.py:318-321) in device memory with a
    lazily synchronised host mirror."""

    def __init__(self, dev: Device, n: int, block_sizes=None, kind=None):
        self.dev = dev
        self.n = int(n)
        self.d = dev.empty(n, np.float64)
        self.d.zero()
        self.block_sizes = list(block_sizes) if block_sizes is not None else [self.n]
        self.kind = kind
        self._host = None
        self._host_valid = False
        self._host_dirty = False  # host copy handed out writable: re-upload before device use
        self._zero_pending = False
        self._prefix = ""

    # device side ------------------------------------------------------------------------
    def device_ptr(self) -> C.c_void_p:
        """Pointer for kernels that READ or UPDATE the vector."""
        self._flush_host()
        if self._zero_pending:
            self.d.zero()
            self._zero_pending = False
        return self.d.c_ptr

    def device_ptr_overwrite(self) -> C.c_void_p:
        """Pointer for kernels that overwrite every entry."""
        self._host_dirty = False
        self._zero_pending = False
        self._host_valid = False
        return self.d.c_ptr

    def mark_device_modified(self) -> None:
        self._host_valid = False

    def _flush_host(self) -> None:
        if self._host_dirty:
            self.d.upload(self._host)
            self._host_dirty = False
            self._zero_pending = False

    # host side --------------------------------------------------------------------------
    def _sync_host(self) -> np.ndarray:
        if self._host is None:
            self._host = self.dev.pinned(self.n)
        if not self._host_valid and not self._host_dirty:
            if self._zero_pending:
                self._host[:] = 0.0
            else:
                self.d.download(self._host)
            self._host_valid = True
        return self._host

    @property
    def array(self) -> np.ndarray:
        """Writable host view (PETSc ``Vec.array``); the device copy is refreshed before next use."""
        h = self._sync_host()
        self._host_dirty = True
        return h

    @property
    def array_r(self) -> np.ndarray:
        h = self._sync_host()
        v = h.view()
        v.flags.writeable = False
        return v

    def getArray(self, readonly: bool = False) -> np.ndarray:
        return self.array_r if readonly else self.array

    def setArray(self, a) -> None:
        self.array[:] = a

    def getSize(self) -> int:
        return self.n

    def getLocalSize(self) -> int:
        return self.n

    size = property(getSize)

    def getType(self) -> str:
        return "nest" if self.kind == "nest" else "seq"

    def getNestSubVecs(self):
        off = np.concatenate([[0], np.cumsum(self.block_sizes)])
        a = self.array_r
        return [a[off[i] : off[i + 1]] for i in range(len(self.block_sizes))]

    def norm(self, norm_type=None) -> float:
        return float(np.linalg.norm(self.array_r))

    def set(self, value: float) -> None:
        if value == 0.0:
            self.zeroEntries()
        else:
            self.array[:] = value

    def zeroEntries(self) -> None:
        """Lazy zero: the assembly kernel overwrites every entry, so no memset is issued unless
        somebody looks at the vector first."""
        self._zero_pending = True
        self._host_dirty = False
        self._host_valid = False

    def copy(self) -> "Vec":
        out = Vec(self.dev, self.n, self.block_sizes, self.kind)
        self.dev.call("nxfx_memcpy_d2d", out.d.c_ptr, self.device_ptr(), C.c_size_t(self.d.nbytes))
        return out

    def duplicate(self) -> "Vec":
        return Vec(self.dev, self.n, self.block_sizes, self.kind)

    def ghostUpdate(self, *args, **kwargs) -> None:
        return None

    def assemble(self) -> None:
        return None

    def setOptionsPrefix(self, prefix: str) -> None:
        self._prefix = prefix

    def getOptionsPrefix(self) -> str:
        return self._prefix

    def setFromOptions(self) -> None:
        return None

    def destroy(self) -> None:
        return None

    def to_petsc(self):
        from petsc4py import PETSc  # noqa: PLC0415

        return PETSc.Vec().createWithArray(self.array_r.copy())


class _Touch:
    """``nxfx_matrix_touch`` of one matrix: the values were written other than by the assembly."""

    def __init__(self, dev: Device, mat_id: int):
        self.dev, self.mat_id = dev, mat_id

    def __call__(self) -> None:
        self.dev.call("nxfx_matrix_bind", C.c_int64(self.mat_id))
        self.dev.call("nxfx_matrix_touch")


class Mat:
    """Monolithic CSR matrix on the pattern of the device context (``nxfx_symbolic``).  Every ``Mat``
    owns its value array (``nxfx_matrix_create``) -- the reference hands out independent PETSc
    matrices (solver.py:43, assembly.py:354), so two solvers / assemblers on one network never alias --
    and binds it before every operation that reads or writes it.

    ``kind`` only changes the reported type and enables ``getNestSubMatrix`` (PETSc MATNEST,
    assembly.py:357); storage is always one CSR so that the SpMV streams a single value array."""

    def __init__(self, dev: Device, n: int, nnz: int, block_sizes, kind=None):
        self.dev = dev
        self.n = int(n)
        self.nnz = int(nnz)
        self.block_sizes = list(block_sizes)
        self.kind = kind
        mid = C.c_int64()
        dev.call("nxfx_matrix_create", C.byref(mid))
        self.mat_id = int(mid.value)
        self._finalizer = weakref.finalize(self, dev.lib.nxfx_matrix_destroy, dev.handle, C.c_int64(self.mat_id))
        self.bind()
        rp, ci, va = C.c_void_p(), C.c_void_p(), C.c_void_p()
        dev.call("nxfx_csr_device", C.byref(rp), C.byref(ci), C.byref(va))
        self.rowptr = DeviceArray(dev, self.n + 1, np.int32, ptr=rp.value)
        self.colidx = DeviceArray(dev, self.nnz, np.int32, ptr=ci.value)
        # a write through Mat.values (upload, zero, or a view's) tells the library (nxfx_matrix_touch); the
        # callback holds the device and the id, not the Mat, so that the Mat is still freed by refcount
        self.values = DeviceArray(dev, self.nnz, np.float64, ptr=va.value, on_write=_Touch(dev, self.mat_id))
        self._zero_pending = True  # a new matrix is zero
        self._pattern_host = None
        self._prefix = ""
        self.assembled = False

    def bind(self) -> None:
        """Make this matrix the target / operator of the following device calls."""
        self.dev.call("nxfx_matrix_bind", C.c_int64(self.mat_id))

    def touch(self) -> None:
        """Declare that the values were written other than by the assembly (a kernel of the caller's own
        through ``values.ptr``, say): the next assembly then writes every entry again.  Writes made through
        ``values.upload`` / ``values.zero`` call this themselves."""
        _Touch(self.dev, self.mat_id)()

    @property
    def static_valid(self) -> bool:
        """True if the values hold the pattern-only entries of an assembly (pressure and multiplier rows),
        which the next overwriting assembly then leaves in place (``nxfx_matrix_static_valid``)."""
        self.bind()
        v = C.c_int32()
        self.dev.call("nxfx_matrix_static_valid", C.byref(v))
        return bool(v.value)

    @property
    def accumulated(self) -> int:
        """Number of assemblies summed into the matrix since it was last zeroed (ADD_VALUES)."""
        self.bind()
        k = C.c_int32()
        self.dev.call("nxfx_matrix_info", None, None, C.byref(k))
        return int(k.value)

    def getSize(self):
        return (self.n, self.n)

    def getLocalSize(self):
        return (self.n, self.n)

    size = property(getSize)

    def getType(self) -> str:
        return "nest" if self.kind == "nest" else "seqaij"

    def zeroEntries(self) -> None:
        """Lazy zero (solver.py:97-98): the next assemble overwrites instead of accumulating."""
        self._zero_pending = True

    def consume_zero(self) -> bool:
        """True if the matrix is (logically) zero, i.e. the assembly may overwrite."""
        z = self._zero_pending
        self._zero_pending = False
        return z

    def zero_now(self) -> None:
        """Write the zeros (values and the solver's per-cell data) and forget the accumulated assemblies."""
        self.bind()
        self.dev.call("nxfx_matrix_zero")
        self.assembled = False

    def _materialise_zero(self) -> None:
        if self._zero_pending and self.assembled:
            self.zero_now()

    def assemble(self) -> None:
        return None

    def setOptionsPrefix(self, prefix: str) -> None:
        self._prefix = prefix

    def getOptionsPrefix(self) -> str:
        return self._prefix

    def setFromOptions(self) -> None:
        return None

    def destroy(self) -> None:
        return None

    def pattern(self):
        if self._pattern_host is None:
            self._pattern_host = (self.rowptr.download(), self.colidx.download())
        return self._pattern_host

    def getValuesCSR(self):
        """(indptr, indices, data) as PETSc returns them (explicit zeros included)."""
        rp, ci = self.pattern()
        if self._zero_pending:
            return rp, ci, np.zeros(self.nnz)
        self.dev.sync()
        return rp, ci, self.values.download()

    def to_scipy(self):
        import scipy.sparse as sp  # noqa: PLC0415

        rp, ci, va = self.getValuesCSR()
        return sp.csr_matrix((va, ci, rp), shape=(self.n, self.n))

    def getNestSubMatrix(self, i: int, j: int):
        """Block (i, j) as a SciPy CSR matrix (host copy; MATNEST view, assembly.py:357)."""
        off = np.concatenate([[0], np.cumsum(self.block_sizes)])
        return self.to_scipy()[off[i] : off[i + 1], off[j] : off[j + 1]]

    def mult(self, x: Vec, y: Vec) -> None:
        """y = A x on the device (CSR-stream SpMV kernel)."""
        self._materialise_zero()
        self.bind()
        self.dev.call("nxfx_spmv", x.device_ptr(), y.device_ptr_overwrite())
        y.mark_device_modified()

    def to_petsc(self):
        from petsc4py import PETSc  # noqa: PLC0415

        rp, ci, va = self.getValuesCSR()
        return PETSc.Mat().createAIJ(size=self.getSize(), csr=(rp, ci, va))


class KSP:
    """Holder of the solver options in PETSc vocabulary (solver.py:41,51-73).  Mapping onto the
    device solver (DESIGN.md "Solver"):

    ============================  =======================================================
    ``ksp_type=preonly, pc=lu``   network Schur-complement direct solve + iterative refinement
    ``ksp_type=gmres|fgmres``     flexible GMRES(restart) with the chosen ``pc_type``
    ``pc_type``                   ``lu``/``cholesky``/``schur`` -> network Schur, ``none``, ``jacobi``
    ============================  =======================================================
    """

    def __init__(self, comm=None):
        self.comm = comm
        self._prefix = ""
        self.options: dict = {}
        self.A = None
        self.its = 0
        self.rnorm = float("nan")
        self.reason = 0
        self.history: list[float] = []

    def setOperators(self, A, P=None) -> None:
        self.A = A

    def getOperators(self):
        return self.A, self.A

    def setOptionsPrefix(self, prefix: str) -> None:
        self._prefix = prefix

    def getOptionsPrefix(self) -> str:
        return self._prefix

    def setFromOptions(self) -> None:
        return None

    def getType(self) -> str:
        return str(self.options.get("ksp_type", "preonly"))

    def getIterationNumber(self) -> int:
        return self.its

    def getResidualNorm(self) -> float:
        return self.rnorm

    def getConvergedReason(self) -> int:
        return self.reason

    def getConvergenceHistory(self):
        return np.asarray(self.history)

    def destroy(self) -> None:
        return None
