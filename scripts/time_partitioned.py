"""Step time of one network cut into parts solved from one process (``PartitionedSolver``) against the same
network solved whole by ``Solver`` on one GPU:

    python scripts/time_partitioned.py [--n 16] [--N 1] [--steps 50] [--devices 0,0] [--exchange peer] [--out FILE]

The step is ``assemble()`` + ``solve()`` (refine_steps=1, the default direct solve).  Each rank times it with the
library's timer entries (``nxfx_timer_start`` / ``nxfx_timer_stop``: CUDA events on the rank's stream); the
partitioned step is the slowest rank's time, next to the host wall clock around the whole step (thread
dispatch included).  Medians over ``--steps`` steps after five warm-up steps.  Prints one JSON line with the card
name and its power limit (and appends it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import networks_fenicsx_b200 as nxfx  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def time_whole(G, N, p_bc, steps):
    nm = nxfx.NetworkMesh(G, N=N)
    asm = nxfx.HydraulicNetworkAssembler(nm)
    asm.compute_forms(p_bc_ex=p_bc)
    solver = nxfx.Solver(asm)
    dev = nm.device
    ms, wall = [], []
    for k in range(5 + steps):
        t0 = time.perf_counter()
        dev.timer_start()
        solver.assemble()
        solver.solve()
        m = dev.timer_stop()
        w = time.perf_counter() - t0
        if k >= 5:
            ms.append(m)
            wall.append(1e3 * w)
    return float(np.median(ms)), float(np.median(wall))


def time_partitioned(G, N, p_bc, steps, devices, exchange):
    with nxfx.PartitionedSolver(G, N, p_bc, devices=devices, exchange=exchange) as ps:
        ms, wall, hist = [], [], None
        for k in range(5 + steps):
            t0 = time.perf_counter()
            ps.map(lambda s: s.dev.timer_start())
            ps.assemble()
            hist = ps.solve()
            per_rank = ps.map(lambda s: s.dev.timer_stop())
            w = time.perf_counter() - t0
            if k >= 5:
                ms.append(max(per_rank))
                wall.append(1e3 * w)
        return ps.exchange, float(np.median(ms)), float(np.median(wall)), hist[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16)
    ap.add_argument("--N", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--devices", default="0,0")
    ap.add_argument("--exchange", default="peer")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    devices = [int(d) for d in a.devices.split(",")]
    G = nxfx.network_generation.make_tree(a.n, a.n, a.n, as_arrays=True)
    p_bc = lambda x: x[1] + 0.1 * x[0]  # noqa: E731
    whole_ms, whole_wall = time_whole(G, a.N, p_bc, a.steps)
    mode, part_ms, part_wall, rel = time_partitioned(G, a.N, p_bc, a.steps, devices, a.exchange)
    rec = {
        "workload": f"make_tree({a.n}) N={a.N}", "edges": G.number_of_edges(), "steps": a.steps,
        "whole_solver_step_ms_median": round(whole_ms, 4), "whole_solver_wall_ms_median": round(whole_wall, 4),
        "devices": devices, "exchange": mode,
        "partitioned_step_ms_median_slowest_rank": round(part_ms, 4),
        "partitioned_wall_ms_median": round(part_wall, 4), "partitioned_relative_residual": rel,
        "gpus": card(),
    }
    line = json.dumps(rec)
    print(line, flush=True)
    if a.out:
        with open(a.out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
