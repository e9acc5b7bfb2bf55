"""The in-process rank harness (tests/inprocess_dist.py) on the CPU: its collectives against what torch.distributed defines,
its failure modes (a bookkeeping mismatch or an error on one rank fails the run instead of hanging it), and the slab
smoothing lengths of distributed.py on three thread-ranks with scipy in place of the CUDA solver, bit-equal to scipy over
the whole set like the gloo test of the same host logic."""
import threading
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist

from inprocess_dist import thread_ranks  # noqa: F401  (fixture)
from test_distributed_cpu import _ScipySolver


SENDS = [[0, 1, 3], [1, 1, 1], [3, 2, 1]]            # rows rank g sends to rank d: SENDS[g][d] (empty and unequal pieces)


def _rows(rank):
    return torch.arange(sum(SENDS[rank]) * 3, dtype=torch.float64).reshape(-1, 3) + 1000 * rank


def test_collectives_follow_torch_distributed(thread_ranks):
    def body(r):
        t = torch.tensor([1.0 + r, 10.0 - r, 100.0 * r])
        s = t.clone(); dist.all_reduce(s, op=dist.ReduceOp.SUM)
        m = t.clone(); dist.all_reduce(m, op=dist.ReduceOp.MIN)
        red = t.clone(); dist.reduce(red, dst=1, op=dist.ReduceOp.SUM)
        parts = [torch.empty(2, dtype=torch.int64) for _ in range(3)]
        dist.all_gather(parts, torch.tensor([r, 7 * r]))
        even_in = torch.arange(6, dtype=torch.int64) + 10 * r                 # 2 rows to every rank
        even_out = torch.empty(6, dtype=torch.int64)
        dist.all_to_all_single(even_out, even_in)
        recv = [SENDS[g][r] for g in range(3)]
        out = torch.empty((sum(recv), 3), dtype=torch.float64)
        dist.all_to_all_single(out, _rows(r), output_split_sizes=recv, input_split_sizes=SENDS[r])
        return s, m, red, parts, even_out, out, dist.get_rank(), dist.get_world_size(), dist.is_initialized()

    res = thread_ranks(3, body)
    vals = [torch.tensor([1.0 + r, 10.0 - r, 100.0 * r]) for r in range(3)]
    for r, (s, m, red, parts, even_out, out, rank, world, init) in enumerate(res):
        assert (rank, world, init) == (r, 3, True)
        assert torch.equal(s, vals[0] + vals[1] + vals[2])
        assert torch.equal(m, torch.minimum(torch.minimum(vals[0], vals[1]), vals[2]))
        assert torch.equal(red, s if r == 1 else vals[r])                    # only dst receives the sum
        assert [p.tolist() for p in parts] == [[g, 7 * g] for g in range(3)]
        assert even_out.tolist() == [v for g in range(3) for v in (10 * g + 2 * r, 10 * g + 2 * r + 1)]
        want = [_rows(g)[sum(SENDS[g][:r]):sum(SENDS[g][:r + 1])] for g in range(3)]
        assert torch.equal(out, torch.cat(want))
    assert not dist.is_initialized()                                          # the calling thread is no rank


def test_all_to_all_rejects_wrong_output_split_sizes(thread_ranks):
    def body(r):
        inp = torch.arange(4, dtype=torch.float64) + 10 * r
        out = torch.empty(4, dtype=torch.float64)
        # each rank sends [1, 3] rows; rank 1 claims it receives [2, 2] (same total, so only the split check can notice)
        dist.all_to_all_single(out, inp, output_split_sizes=[1, 1] if r == 0 else [2, 2], input_split_sizes=[1, 3])

    with pytest.raises(AssertionError, match="received rows"):
        thread_ranks(2, body)


def test_an_error_on_one_rank_fails_the_run_without_hanging(thread_ranks):
    def body(r):
        if r == 2:
            raise ValueError("rank 2 gives up")
        t = torch.ones(1)
        dist.all_reduce(t)                                                    # ranks 0, 1, 3 wait here for rank 2
        dist.all_reduce(t)

    t0 = time.perf_counter()
    with pytest.raises(ValueError, match="rank 2 gives up"):
        thread_ranks(4, body)
    assert time.perf_counter() - t0 < 30.0                                    # the barrier was aborted, not timed out
    assert not [t for t in threading.enumerate() if t.name.startswith("inprocess-rank-")]


def _slab_scene(case):
    from astro_sph_tools_b200 import distributed as astd, synthetic
    if case == "lattice_periodic":
        pos, _ = synthetic.s1_positions(20); box, k = 1.0, 16
    elif case.startswith("clustered_periodic"):
        pos, _ = synthetic.s2_positions(6000, 1.0, n_haloes=4, seed=3); box, k = 1.0, 24
    else:                                                                     # open box, random order
        rng = np.random.default_rng(9); pos = rng.normal(size=(5000, 3)) * np.array([3.0, 1.0, 0.5]); box, k = None, 12
    n = len(pos)
    cuts = [0, (n * 2) // 5, (n * 3) // 4, n] if case == "open_unequal" else [astd.shard_bounds(n, 3, r)[0] for r in range(3)] + [n]
    return pos, box, k, cuts


@pytest.mark.parametrize("case,ghost_width", [("lattice_periodic", None), ("clustered_periodic", None),
                                              ("clustered_periodic", 0.01), ("open_unequal", None)])
def test_slab_smoothing_lengths_on_thread_ranks_equal_the_full_search(thread_ranks, oracle, case, ghost_width):
    """the scenes of test_slab_ghost_smoothing_lengths_equal_the_full_search on 3 thread-ranks; with ghost_width = 0.01 the
    clustered set widens its ghost zone several times and two ranks end up holding nearly the whole set"""
    from astro_sph_tools_b200 import distributed as astd
    pos, box, k, cuts = _slab_scene(case)

    def body(r):
        return astd.smoothing_lengths_slabs(torch.from_numpy(pos[cuts[r]:cuts[r + 1]].copy()), k, box, solver=_ScipySolver(),
                                            ghost_width=ghost_width, return_stats=True)

    res = thread_ranks(3, body)
    ref = oracle.knn_scipy(pos, k, box)[0]
    for r, (h, st) in enumerate(res):
        assert np.array_equal(h.numpy(), ref[cuts[r]:cuts[r + 1]]), f"rank {r}"
    assert sum(st["owned"] for _, st in res) == len(pos)
    if case == "lattice_periodic":
        assert all(st["local_set"] < 0.95 * len(pos) for _, st in res)
    if ghost_width:
        assert all(st["iterations"] >= 2 for _, st in res)
        assert max(st["local_set"] for _, st in res) > 2 * max(st["owned"] for _, st in res)


def test_sharded_smoothing_lengths_on_thread_ranks(thread_ranks, oracle):
    """replicated positions (one all-gather of unequal shards), every rank answers its own index range"""
    from astro_sph_tools_b200 import distributed as astd
    pos = np.random.default_rng(5).uniform(0, 1, (2003, 3))
    cuts = [0, 700, 710, 2003]
    res = thread_ranks(3, lambda r: astd.smoothing_lengths_sharded(torch.from_numpy(pos[cuts[r]:cuts[r + 1]].copy()), 16, 1.0,
                                                                   solver=_ScipySolver()))
    ref = oracle.knn_scipy(pos, 16, 1.0)[0]
    for r, h in enumerate(res):
        assert np.array_equal(h.numpy(), ref[cuts[r]:cuts[r + 1]])
