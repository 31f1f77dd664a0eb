"""Time the assembly and the back-substitution of the headline workload (development helper).

    python scripts/time_assembly.py [generations] [repetitions]

Three figures at make_tree(generations), N = 1, P1/DG0, each the mean over the repetitions after one warm-up call:
  full write   nxfx_assemble (matrix + rhs) that writes every matrix entry: a fresh matrix, or one after
               zero_now / a write through its values.  Here nxfx_matrix_touch before every call (host flag only,
               nothing is launched) forces it.
  re-assembly  the same call repeated on the matrix it assembled last, as Solver.assemble() runs every step:
               the pressure rows {-1, +1} and the multiplier rows (0, +1) / (-1, 0) stay where they are.
  back-subst.  edge_backsub_n1_kernel as nxfx_pc_apply launches it after the stored-factor tree solve: kernel
               durations from torch.profiler (CUPTI) over the repetitions, in a pass of its own after the event
               timings.  (Inside nxfx_solve it is a programmatic dependent of the tree kernel: it starts while that
               kernel drains and waits for it, so its duration there is not its cost.)
The bytes are the ones each kernel moves to or from HBM: vertex records (32 per vertex), slot records, the
values it writes, b, R*h; for the back-substitution r, R*h, the slot records and z (the multipliers it gathers
are L2-resident and not counted).  The working set (~0.2 GB) is larger than the 126 MB L2: no flush is needed
between the timed calls.
"""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
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
dev, A = nm.device, solver.A
A.bind()
bb = solver.b.duplicate()
R_d, R_c = asm._R
f_d, f_c = asm._f


def assemble():
    dev.call("nxfx_assemble", R_d.c_ptr if R_d is not None else None, C.c_double(R_c),
             f_d.c_ptr if f_d is not None else None, C.c_double(f_c), 1, 1, 0, bb.d.c_ptr)


def full_write():
    dev.call("nxfx_matrix_touch")
    assemble()


def timeit(fn):
    fn(); dev.sync(); dev.timer_start()
    for _ in range(reps):
        fn()
    return dev.timer_stop() / reps * 1e3  # us


t_full = timeit(full_write)
t_re = timeit(assemble)
skips = A.static_valid

# byte counts from the sizes of this network
E = nm.graph_edges.shape[0]
nv = nm.mesh.topology.index_map(0).size_local
n_bif = nm.bifurcation_values.size
nd, nnz = asm.num_dofs, A.nnz
rp = A.pattern()[0]
nq = sum(asm.block_sizes[:-2])
n_static = int(rp[-1] - rp[nq])  # entries of the pressure and multiplier rows
reads = 32 * nv + 8 * E  # vertex records, 8-byte slot records {u, v}
writes = 8 * nnz + 8 * nd + 8 * E  # values, b, R*h
b_full = reads + writes
b_re = b_full - 8 * n_static if skips else b_full
b_alg = 24 * nv + 8 * nnz + 8 * nd + 8 * nm.boundary_values.size  # bench.py roofline_assembly (full write)
b_bs = E * (8 + 4 + 24 + 8 + 24) + 16 * n_bif  # {lm(u), lm(v)}, slot_edge, r, R*h, z per slot; lam -> z

# back-substitution: kernel durations of preconditioner applications with the stored factors
z = solver.b.duplicate()
bp, zp = solver.b.d.c_ptr, z.d.c_ptr
t_bs, n_bs = None, 0
try:
    from torch.profiler import ProfilerActivity, profile

    dev.call("nxfx_pc_setup")
    dev.call("nxfx_pc_apply", bp, zp); dev.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            dev.call("nxfx_pc_apply", bp, zp)
        dev.sync()
    durs = [e.time_range.elapsed_us() for e in prof.events() if "edge_backsub_n1_kernel" in e.name]
    if durs:
        t_bs, n_bs = sum(durs) / len(durs), len(durs)
except Exception as e:  # the event timings above stand without it
    print(f"torch.profiler pass failed: {e}")

try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
except Exception as e:  # the timings stand without it, the card is printed as unknown
    card = f"unknown ({e})"
print(f"card {card}")
print(f"make_tree({n}) N=1  n_dofs {nd}  nnz {nnz}  pressure + multiplier entries {n_static} "
      f"({8 * n_static / 1e6:.1f} MB)  repetitions {reps}")
print(f"  {'assembly, full write':34s} {t_full:7.2f} us  {b_full / 1e6:7.1f} MB  {b_full / t_full / 1e3:7.0f} GB/s")
print(f"  {'assembly, re-assembly' + ('' if skips else ' (writes every entry)'):34s} {t_re:7.2f} us  "
      f"{b_re / 1e6:7.1f} MB  {b_re / t_re / 1e3:7.0f} GB/s")
print(f"  {'(bench.py algorithmic, full write)':34s} {'':10s}  {b_alg / 1e6:7.1f} MB")
if t_bs is not None:
    print(f"  {'back-substitution (profiler)':34s} {t_bs:7.2f} us  {b_bs / 1e6:7.1f} MB  {b_bs / t_bs / 1e3:7.0f} GB/s  "
          f"({n_bs} launches)")
else:
    print("  back-substitution: not measured (no profiler events)")
