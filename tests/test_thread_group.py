"""CPU checks of the in-process collectives (``ThreadGroup``) and of the worker threads of ``PartitionedSolver``:
sums in rank order, identical on every rank; a rank that raises breaks the barrier of the others; a failing
rank's exception reaches the caller with every thread joined."""

import threading

import numpy as np
import pytest
import torch

from networks_fenicsx_b200.distributed import PartitionedSolver, ThreadGroup


def run_ranks(world, fn, timeout=60.0):
    """fn(group) on ``world`` plain threads; (results, exceptions) in rank order."""
    groups = ThreadGroup.create(world, timeout=timeout)
    results, errors = [None] * world, [None] * world

    def body(r):
        try:
            results[r] = fn(groups[r])
        except BaseException as exc:  # noqa: BLE001 -- reported to the test
            groups[r].abort()
            errors[r] = exc

    threads = [threading.Thread(target=body, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=2 * timeout)
    assert not any(t.is_alive() for t in threads)
    return results, errors


def test_all_reduce_sums_in_rank_order():
    world = 4
    # chosen so that the order of the additions shows: (1e16 + 1) + (-1e16) + 1 != 1e16 + (-1e16) + 1 + 1
    vals = np.array([[1e16, 0.5], [1.0, 0.25], [-1e16, 3.0], [1.0, -0.125]])
    expect = vals[0].copy()
    for v in vals[1:]:
        expect = expect + v

    def fn(g):
        t = torch.tensor(vals[g.rank], dtype=torch.float64)
        g.all_reduce(t)
        s = g.all_reduce_scalar(vals[g.rank, 0])
        out = [torch.empty(2, dtype=torch.uint8) for _ in range(g.world)]
        g.all_gather(out, torch.tensor([g.rank, 7 * g.rank], dtype=torch.uint8))
        objs = g.gather_object(("rank", g.rank))
        g.barrier()
        return t.numpy(), s, [o.tolist() for o in out], objs

    results, errors = run_ranks(world, fn)
    assert errors == [None] * world
    assert not np.array_equal(expect, vals[[0, 2, 1, 3]].sum(axis=0))  # the order matters for these values
    for t, s, gathered, objs in results:
        assert np.array_equal(t, expect)  # bit-identical, rank order
        assert s == expect[0]
        assert gathered == [[r, 7 * r] for r in range(world)]
        assert objs == [("rank", r) for r in range(world)]


def test_repeated_collectives_do_not_mix_rounds():
    """Back-to-back collectives reuse the two slot rounds: every call sees its own values."""

    def fn(g):
        return [g.all_reduce_scalar(10 * k + g.rank) for k in range(50)]

    results, errors = run_ranks(3, fn)
    assert errors == [None] * 3
    for res in results:
        assert res == [float(30 * k + 3) for k in range(50)]


def test_a_failing_rank_releases_the_barrier():
    world = 4
    entered = threading.Event()

    def fn(g):
        if g.rank == 2:
            entered.wait(10)
            raise ValueError("rank 2 failed")
        if g.rank == 0:
            entered.set()
        g.all_reduce(torch.zeros(3, dtype=torch.float64))  # would wait for rank 2 until the timeout
        return "finished"

    results, errors = run_ranks(world, fn, timeout=120.0)
    assert isinstance(errors[2], ValueError)
    for r in (0, 1, 3):
        assert isinstance(errors[r], threading.BrokenBarrierError), errors[r]


def test_partitioned_solver_reraises_with_every_thread_joined():
    """Without a GPU every rank fails to set its device up: the caller gets the exception, and the
    worker threads are gone."""
    if torch.cuda.is_available():
        pytest.skip("GPU present (the GPU tests cover the solver)")
    import networks_fenicsx_b200 as nxfx

    G = nxfx.network_generation.make_tree(6, 6, 6, as_arrays=True)
    before = set(threading.enumerate())
    with pytest.raises(Exception) as info:
        PartitionedSolver(G, 1, lambda x: x[1], devices=[0, 0, 0], timeout=30.0)
    assert not isinstance(info.value, threading.BrokenBarrierError)
    left = [t for t in threading.enumerate() if t not in before and t.name.startswith("nxfx-rank")]
    assert left == []
