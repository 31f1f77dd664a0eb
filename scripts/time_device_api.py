"""Step time of the public API with host buffers against the same loop with CUDA tensors, and the bare device step:

    python scripts/time_device_api.py [--n 20] [--steps 500] [--warmup 50] [--rounds 2] [--out FILE]

make_tree(n), one cell per edge, P1/DG0, p_bc(x) = x[1], R = 1, f = 0 (bench.py's tree workload):

  (a) host   ``compute_forms(pinned p_bc array)`` + ``Solver.assemble()`` + ``Solver.solve(create_functions())``:
             bench.py's ``e2e`` loop (p_bc runs up, the solution down into the pinned functions);
  (b) device p_bc evaluated on the GPU from ``NetworkMesh.vertex_coordinates_device()`` (one torch copy per step),
             ``compute_forms(p_bc tensor)`` + ``assemble()`` + ``solve(create_functions(device=True))``;
  (c) bare   ``Solver.assemble()`` + ``nxfx_solve`` into ``solver.x``: the device step of bench.py;
  (d) copy   the device-to-device copy of the solution into ``solver.x`` that every solve of (b) makes, alone.

Each loop is timed with CUDA events on the current torch stream (the library's stream, the legacy default one) over
``--steps`` steps after ``--warmup`` steps, and the host wall clock around the same window; the loops run one after
the other, ``--rounds`` times.  Host<->device bytes of one step are counted from the library calls the step makes
(``nxfx_memcpy_h2d`` / ``nxfx_memcpy_d2h`` sizes, plus the solution mirror of ``create_functions()``).  Prints one
JSON line with the card name and its power limit (and appends it to --out)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import networks_fenicsx_b200 as nxfx  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()


class ByteCounter:
    """Wraps ``Device.call`` and adds up the bytes the calls move between host and device."""

    def __init__(self, dev, n_dofs):
        self.dev, self.n_dofs, self._call = dev, n_dofs, dev.call
        self.h2d = self.d2h = 0

    def __call__(self, name, *args):
        if name in ("nxfx_memcpy_h2d", "nxfx_memcpy_d2h"):
            nbytes = args[-1].value if isinstance(args[-1], C.c_size_t) else int(args[-1])
            if name.endswith("h2d"):
                self.h2d += nbytes
            else:
                self.d2h += nbytes
        elif name == "nxfx_set_solution_mirror" and args[0] is not None:
            self.d2h += 8 * self.n_dofs  # the library copies x into the pinned functions
        return self._call(name, *args)

    def count(self, step):
        self.dev.call = self
        try:
            step()
        finally:
            del self.dev.call
        torch.cuda.synchronize()
        return {"h2d": self.h2d, "d2h": self.d2h}


def timed(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    e1.synchronize()
    wall = time.perf_counter() - t0
    return {"ms_per_step_events": e0.elapsed_time(e1) / steps, "ms_per_step_wall": 1e3 * wall / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=20)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("time_device_api.py measures on a CUDA device; there is none")

    G = nxfx.network_generation.make_tree(args.n, args.n, args.n, as_arrays=True)
    nm = nxfx.NetworkMesh(G, N=1, color_strategy="smallest_last")
    asm = nxfx.HydraulicNetworkAssembler(nm)
    asm.compute_forms(p_bc_ex=lambda x: x[1])
    solver = nxfx.Solver(asm)
    dev = nm.device
    n_dofs = asm.num_dofs
    pbc_pinned = dev.pinned(asm._pbc_host.size)
    pbc_pinned[:] = asm._pbc_host
    fns_host = solver.create_functions()
    X = nm.vertex_coordinates_device()
    pbc_t = torch.empty(X.shape[0], dtype=torch.float64, device=X.device)
    fns_dev = solver.create_functions(device=True)
    opts, info = solver.solve_options(), nxfx._lib.SolveInfo()

    def host_step():
        asm.compute_forms(p_bc_ex=pbc_pinned)
        solver.assemble()
        solver.solve(fns_host)

    def device_step():
        pbc_t.copy_(X[:, 1])  # p_bc(x) = x[1] evaluated on the GPU
        asm.compute_forms(p_bc_ex=pbc_t)
        solver.assemble()
        solver.solve(fns_dev)

    def bare_step():
        solver.assemble()
        dev.call("nxfx_solve", solver.b.device_ptr(), solver.x.device_ptr_overwrite(), C.byref(opts), C.byref(info))

    def copy_into_x():  # the part of (b)'s solve that keeps solver.x holding the solution
        dev.call("nxfx_memcpy_d2d", solver.x.device_ptr_overwrite(), fns_dev[0]._device_buffer.c_ptr,
                 C.c_size_t(8 * n_dofs))

    loops = {"a_host_buffers": host_step, "b_device_tensors": device_step, "c_bare_device_step": bare_step,
             "d_solution_copy_into_solver_x": copy_into_x}
    host_step()
    x_host = np.concatenate([fn.x.array for fn in fns_host])
    device_step()
    same = bool(np.array_equal(torch.cat([fn.x.array for fn in fns_dev]).cpu().numpy(), x_host))
    rounds = []
    for _ in range(args.rounds):
        rounds.append({name: timed(step, args.steps, args.warmup) for name, step in loops.items()})
    bytes_per_step = {name: ByteCounter(dev, n_dofs).count(step) for name, step in loops.items()}
    res = {
        "what": f"make_tree({args.n}), N=1, P1/DG0, p_bc = x[1]: API step with host buffers (a), with CUDA tensors (b), "
                "bare device step (c), the copy of the solution into solver.x that (b) makes (d)",
        "card": card(),
        "n_dofs": n_dofs,
        "steps": args.steps,
        "warmup": args.warmup,
        "rounds": rounds,
        "bytes_per_step": bytes_per_step,
        "device_solution_equals_host_solution": same,
        "torch": torch.__version__,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
