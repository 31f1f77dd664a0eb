"""Time the CSR products of the headline workload with CUDA events (development helper).

    NXFX_LIB=/path/to/variant.so python scripts/time_residual.py [generations] [repetitions]

Three figures, each the mean over the repetitions after one warm-up call:
  spmv      y = A x                        (nxfx_spmv)
  residual  r = b - A x, r written         (nxfx_residual without the norm read-back)
  in-step   the norms-only residual check inside nxfx_solve, which no ABI call runs alone: the step with
            the default options (fresh matrix: nxfx_assemble + nxfx_solve) minus the same pair with
            refine_steps = 0 and final_residual = 0 (the plain application, no residual check)
The bytes are those streamed from HBM: values and columns (12 per entry), row pointers, b where it is read
and the written vector; x (8 n, gathered from L2 after the first touch) is listed apart.
"""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from networks_fenicsx_b200 import _lib  # noqa: E402

if os.environ.get("NXFX_LIB"):
    import pathlib

    _lib.LIB_PATH = pathlib.Path(os.environ["NXFX_LIB"])
import networks_fenicsx_b200 as nxfx  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 20
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 200
G = nxfx.network_generation.make_tree(n, n, n, as_arrays=True)
nm = nxfx.NetworkMesh(G, N=1, color_strategy="smallest_last")
asm = nxfx.HydraulicNetworkAssembler(nm)
asm.compute_forms(p_bc_ex=lambda x: x[1])
solver = nxfx.Solver(asm)
solver.assemble()
solver.solve()
dev = nm.device
nnz, nd = solver.A.nnz, asm.num_dofs


def timeit(fn, k=reps):
    fn(); dev.sync(); dev.timer_start()
    for _ in range(k):
        fn()
    return dev.timer_stop() / k * 1e3  # us


y = solver.b.duplicate(); bb = solver.b.duplicate()
xp, yp, bp = solver.x.d.c_ptr, y.d.c_ptr, solver.b.d.c_ptr
t_spmv = timeit(lambda: dev.call("nxfx_spmv", xp, yp))
t_res = timeit(lambda: dev.call("nxfx_residual", bp, xp, yp, None))
info = _lib.SolveInfo()
full = solver.solve_options()
plain = solver.solve_options()
plain.refine_steps = 0
plain.final_residual = 0


def step(opts):
    dev.call("nxfx_assemble", None, C.c_double(1.0), None, C.c_double(0.0), 1, 1, 0, bb.d.c_ptr)
    dev.call("nxfx_solve", bp, xp, C.byref(opts), C.byref(info))


k_step = max(reps // 4, 20)
t_full, t_plain = [], []
for _ in range(5):  # interleaved: both arms see the same clock and neighbours
    t_full.append(timeit(lambda: step(full), k_step))
    t_plain.append(timeit(lambda: step(plain), k_step))
t_full.sort(); t_plain.sort()
t_instep = t_full[2] - t_plain[2]

mat = 12 * nnz + 4 * (nd + 1)
rows = [("spmv y = A x", t_spmv, mat + 8 * nd),
        ("residual r = b - A x", t_res, mat + 16 * nd),
        ("in-step norms-only residual", t_instep, mat + 8 * nd)]
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
except Exception as e:  # the timings stand without it, the card is printed as unknown
    card = f"unknown ({e})"
print(f"library {os.environ.get('NXFX_LIB', 'default')}  card {card}")
print(f"generations {n}  n_dofs {nd}  nnz {nnz}  x {8 * nd / 1e6:.1f} MB (L2, not counted)")
for name, t, b in rows:
    print(f"  {name:30s} {t:7.2f} us  {b / 1e6:7.1f} MB  {b / t / 1e3:7.0f} GB/s")
print(f"  step with check {t_full[2]:7.2f} us (range {t_full[0]:.2f}-{t_full[-1]:.2f}), "
      f"without {t_plain[2]:7.2f} us (range {t_plain[0]:.2f}-{t_plain[-1]:.2f})")
