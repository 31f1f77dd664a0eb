"""Weak scaling of the higher-order direct solve on a partitioned network (host-driven exchange, NCCL):

    torchrun --nproc-per-node W scripts/time_generic_dist.py [--base 16] [--N 4] [--steps 20] [--out FILE]

Each of the W ranks (one GPU each) holds about one make_tree(base) worth of edges: the whole network is
make_tree(base + log2 W).  For P2/P1 and P3/P2 the step -- factorisation + first application (one all-reduce),
the residual (one all-reduce) -- is timed with CUDA events over ``--steps`` steps after two warm-up steps, and
the all-reduces are bracketed with CUDA events of their own to give their share of the step.  Rank 0 prints one
JSON line per degree pair (and appends it to --out) with the card name and its power limit.  Ranks that share
a GPU time-slice, so the script refuses more ranks than devices."""
import argparse
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import networks_fenicsx_b200 as nxfx  # noqa: E402
from networks_fenicsx_b200.distributed import DistributedSolver  # noqa: E402


class TimedCollectives:
    """The solver's collectives with every all_reduce bracketed by CUDA events (summed per step)."""

    def __init__(self, inner):
        self.inner = inner
        self.pairs = []

    def __getattr__(self, name):
        return getattr(self.inner, name)

    def all_reduce(self, t):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        self.inner.all_reduce(t)
        b.record()
        self.pairs.append((a, b))

    def take_ms(self):
        ms = sum(a.elapsed_time(b) for a, b in self.pairs)
        self.pairs = []
        return ms


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", type=int, default=16)
    ap.add_argument("--N", type=int, default=4)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > torch.cuda.device_count():
        raise SystemExit(f"{world} ranks on {torch.cuda.device_count()} GPU(s): ranks sharing a GPU are not a measurement")
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rank = dist.get_rank()
    n = a.base + int(round(math.log2(world)))
    G = nxfx.network_generation.make_tree(n, n, n, as_arrays=True)
    for fd, pd in ((2, 1), (3, 2)):
        ds = DistributedSolver(G, a.N, lambda x: x[1] + 0.1 * x[0], device=local_rank, exchange="nccl",
                               flux_degree=fd, pressure_degree=pd)
        coll = ds._comm = TimedCollectives(ds._comm)
        ds.assemble()
        for _ in range(2):
            ds.solve(refine_steps=0, final_residual=True)
        coll.take_ms()
        steps, shares = [], []
        for _ in range(a.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            hist = ds.solve(refine_steps=0, final_residual=True)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            steps.append(ms)
            shares.append(coll.take_ms() / ms)
        t = torch.tensor([np.median(steps), np.median(shares)], dtype=torch.float64, device="cuda")
        gathered = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        if rank == 0:
            per_rank = [g.cpu().numpy().tolist() for g in gathered]
            rec = {
                "workload": f"make_tree({n}) N={a.N} P{fd}/P{pd}", "world": world, "n_dofs": ds.n_dofs_global,
                "n_shared": ds.part.n_top, "edges_per_rank": int(G.number_of_edges() / world),
                "step_ms_median_max_over_ranks": max(p[0] for p in per_rank),
                "allreduce_share_median_per_rank": [round(p[1], 4) for p in per_rank],
                "relative_residual": hist[-1], "steps": a.steps, "gpus": card(),
            }
            line = json.dumps(rec)
            print(line, flush=True)
            if a.out:
                with open(a.out, "a") as fh:
                    fh.write(line + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
