"""ctypes binding of the C ABI declared in ``include/nxfx_b200.h``.

There is no CPU fallback: if the shared library is missing or no CUDA device is usable, every
entry point raises ``RuntimeError``.
"""

from __future__ import annotations

import ctypes as C
import pathlib

LIB_PATH = pathlib.Path(__file__).parent / "csrc" / "libnxfx_b200.so"
HISTORY_LEN = 128

c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)


class SolveOpts(C.Structure):
    _fields_ = [
        ("ksp_type", C.c_int32),
        ("pc_type", C.c_int32),
        ("rtol", C.c_double),
        ("atol", C.c_double),
        ("max_it", C.c_int32),
        ("restart", C.c_int32),
        ("refine_steps", C.c_int32),
        ("error_if_not_converged", C.c_int32),
        ("final_residual", C.c_int32),
        ("reserved", C.c_int32),
        ("refine_rtol", C.c_double),
    ]


class SolveInfo(C.Structure):
    _fields_ = [
        ("iterations", C.c_int32),
        ("converged", C.c_int32),
        ("rhs_norm", C.c_double),
        ("residual_norm", C.c_double),
        ("history_len", C.c_int32),
        ("history", C.c_double * HISTORY_LEN),
    ]


KSP_PREONLY, KSP_FGMRES = 0, 1
PC_NETWORK_SCHUR, PC_NONE, PC_JACOBI_FLUX = 0, 1, 2

# name -> (restype, argtypes); every symbol of include/nxfx_b200.h
SIGNATURES = {
    "nxfx_abi_version": (C.c_int, []),
    "nxfx_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "nxfx_destroy": (C.c_int, [C.c_void_p]),
    "nxfx_last_error": (C.c_char_p, [C.c_void_p]),
    "nxfx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_sync": (C.c_int, [C.c_void_p]),
    "nxfx_launch_count": (C.c_int64, [C.c_void_p]),
    "nxfx_malloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "nxfx_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_host_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "nxfx_host_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "nxfx_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "nxfx_memcpy_d2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "nxfx_memset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t]),
    "nxfx_timer_start": (C.c_int, [C.c_void_p]),
    "nxfx_timer_stop": (C.c_int, [C.c_void_p, c_f64p]),
    "nxfx_set_network": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_f64p, c_i32p, c_i32p, c_i32p,
         c_i32p, C.c_int32, c_i32p, c_i32p],
    ),
    "nxfx_update_node_positions": (C.c_int, [C.c_void_p, c_f64p]),
    "nxfx_get_sizes": (
        C.c_int,
        [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
         C.POINTER(C.c_int64)],
    ),
    "nxfx_mesh_geometry_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "nxfx_symbolic": (C.c_int, [C.c_void_p]),
    "nxfx_csr_device": (
        C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    ),
    "nxfx_matrix_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "nxfx_matrix_destroy": (C.c_int, [C.c_void_p, C.c_int64]),
    "nxfx_matrix_bind": (C.c_int, [C.c_void_p, C.c_int64]),
    "nxfx_matrix_zero": (C.c_int, [C.c_void_p]),
    "nxfx_matrix_info": (
        C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    ),
    "nxfx_set_boundary_pressure": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_assemble": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int,
         C.c_void_p],
    ),
    "nxfx_set_tree_schedule": (
        C.c_int,
        [C.c_void_p, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, C.c_int32, c_i32p, C.c_int32, c_i32p,
         C.c_int32, c_i32p],
    ),
    "nxfx_pc_setup": (C.c_int, [C.c_void_p]),
    "nxfx_pc_apply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_spmv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_residual": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_f64p]),
    "nxfx_solve": (
        C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SolveOpts), C.POINTER(SolveInfo)]
    ),
    "nxfx_set_solution_mirror": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_assemble_solve_host": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.POINTER(SolveOpts),
         C.c_void_p, C.POINTER(SolveInfo)],
    ),
    "nxfx_set_generic_system": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, c_i32p, c_i32p, c_i32p, c_f64p, c_i32p, c_i32p, c_f64p],
    ),
    "nxfx_assemble_generic": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_int, C.c_int, C.c_int, C.c_void_p],
    ),
    "nxfx_set_condensation": (
        C.c_int,
        [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_i32p, c_i32p, c_i32p, c_i32p,
         c_i32p, c_i32p, c_i32p, c_i32p, c_f64p, c_i32p, c_i32p, c_i32p, c_f64p, c_i32p, c_i32p, c_i32p, c_f64p, c_i32p],
    ),
    "nxfx_set_shared": (C.c_int, [C.c_void_p, C.c_int32, c_i32p, c_f64p]),
    "nxfx_comm_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_int32)]),
    "nxfx_comm_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_comm_connect_local": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32]),
    "nxfx_comm_destroy": (C.c_int, [C.c_void_p]),
    "nxfx_group_sum": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_void_p, C.c_int64]),
    "nxfx_exchange_sizes": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "nxfx_pc_setup_begin": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_pc_setup_end": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nxfx_pc_apply_begin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_pc_apply_end": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "nxfx_pc_setup_apply_begin": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_pc_setup_apply_end": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_residual_partial": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_residual_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nxfx_global_flux": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load libnxfx_b200.so and declare every prototype.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  networks_fenicsx_b200 has no CPU fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.nxfx_abi_version() != 2:
        raise RuntimeError("libnxfx_b200.so ABI version mismatch")
    _lib = lib
    return lib


def as_i32p(a):
    return a.ctypes.data_as(c_i32p)


def as_f64p(a):
    return a.ctypes.data_as(c_f64p)
