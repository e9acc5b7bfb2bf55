"""In-process ranks for the multi-GPU code of distributed.py: `world` threads of one process play the ranks, and a small
stand-in for the torch.distributed calls that module makes moves tensors between them with plain torch copies.  The
production code then runs unchanged, with its real CUDA kernels, on one device (or on CPU tensors).

A collective works in three steps: every rank posts its tensor in a shared slot and waits on a barrier; every rank builds
its result from clones of the slots; a second barrier keeps any slot from being reused before every rank has read it.
All threads use the device's default stream, so a clone a rank enqueues is ordered after the kernels that produced the
slot on another rank (they were enqueued before the first barrier) and before anything that rank enqueues after the second.

Nothing outlives a run: there is no process group, no process, no NCCL, and every thread is joined.  Use it through the
`thread_ranks` fixture:  `thread_ranks(world, fn)` runs fn(rank) on every rank and returns the results in rank order; an
error on any rank is raised again in the calling thread."""
import threading

import pytest
import torch
import torch.distributed as dist

PATCHED = ("is_available", "is_initialized", "get_world_size", "get_rank", "all_reduce", "reduce", "all_gather",
           "all_to_all_single")
THREAD_PREFIX = "inprocess-rank-"


def _reduce(tensors, op):
    acc = tensors[0].clone()
    for t in tensors[1:]:
        if op == dist.ReduceOp.SUM:
            acc += t
        elif op == dist.ReduceOp.MIN:
            acc = torch.minimum(acc, t)
        else:
            raise NotImplementedError(f"reduce op {op}")
    return acc


class InProcessRanks:
    """The torch.distributed functions distributed.py calls, for ranks that are threads of this process."""

    def __init__(self, timeout=120.0):
        self.timeout = timeout
        self.world = 0
        self._local = threading.local()
        self._barrier = None
        self._slots = []

    def install(self, monkeypatch):
        for name in PATCHED:
            monkeypatch.setattr(dist, name, getattr(self, name))

    # ---- group queries: a thread started by run() is a rank, any other thread sees no process group
    def is_available(self):
        return True

    def is_initialized(self):
        return hasattr(self._local, "rank")

    def get_world_size(self, group=None):
        return self.world

    def get_rank(self, group=None):
        return self._local.rank

    # ---- collectives
    def _collective(self, value, read):
        """post `value`, then return read(every rank's value in rank order); read must copy what it keeps"""
        self._slots[self._local.rank] = value
        self._barrier.wait()
        out = read(self._slots)
        self._barrier.wait()
        return out

    def all_reduce(self, tensor, op=dist.ReduceOp.SUM, group=None, async_op=False):
        assert not async_op
        tensor.copy_(self._collective(tensor, lambda slots: _reduce(slots, op)))

    def reduce(self, tensor, dst, op=dist.ReduceOp.SUM, group=None, async_op=False):
        assert not async_op
        me = self._local.rank
        acc = self._collective(tensor, lambda slots: _reduce(slots, op) if me == dst else None)
        if me == dst:
            tensor.copy_(acc)

    def all_gather(self, tensor_list, tensor, group=None, async_op=False):
        assert not async_op and len(tensor_list) == self.world
        parts = self._collective(tensor, lambda slots: [t.clone() for t in slots])
        for out, part in zip(tensor_list, parts):
            assert out.shape == part.shape, f"all_gather: {tuple(part.shape)} into {tuple(out.shape)}"
            out.copy_(part)

    def all_to_all_single(self, output, input, output_split_sizes=None, input_split_sizes=None, group=None, async_op=False):
        assert not async_op
        w, me = self.world, self._local.rank
        if input_split_sizes is None:
            assert input.shape[0] % w == 0
            input_split_sizes = [input.shape[0] // w] * w
        if output_split_sizes is None:
            assert output.shape[0] % w == 0
            output_split_sizes = [output.shape[0] // w] * w
        sends = [int(s) for s in input_split_sizes]
        assert len(sends) == w and sum(sends) == input.shape[0], f"rank {me}: input splits {sends} of {input.shape[0]} rows"

        def read(slots):
            pieces = []
            for src_input, splits in slots:
                begin = sum(splits[:me])
                pieces.append(src_input[begin:begin + splits[me]].clone())
            return pieces

        pieces = self._collective((input, sends), read)
        got = [p.shape[0] for p in pieces]
        # a mismatch in the caller's bookkeeping fails here instead of being papered over by a reshape
        assert got == [int(s) for s in output_split_sizes], f"rank {me}: received rows {got}, output_split_sizes {list(output_split_sizes)}"
        recv = torch.cat(pieces)
        assert recv.shape == output.shape, f"rank {me}: received {tuple(recv.shape)} into {tuple(output.shape)}"
        output.copy_(recv)

    # ---- running the ranks
    def run(self, world, fn):
        """fn(rank) on `world` threads; returns the results in rank order, re-raises the first error of any rank"""
        self.world = world
        self._barrier = threading.Barrier(world, timeout=self.timeout)
        self._slots = [None] * world
        results = [None] * world
        errors = []
        lock = threading.Lock()

        def body(rank):
            self._local.rank = rank
            try:
                results[rank] = fn(rank)
            except BaseException as e:                    # the others fail at their next barrier instead of hanging
                with lock:
                    errors.append((rank, e))
                self._barrier.abort()

        threads = [threading.Thread(target=body, args=(r,), name=f"{THREAD_PREFIX}{r}", daemon=True) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join(self.timeout * 4)
        alive = [t.name for t in threads if t.is_alive()]
        if alive:
            self._barrier.abort()
            for t in threads:
                t.join(self.timeout)
            raise RuntimeError(f"ranks still running after {self.timeout * 4:.0f} s: {alive}")
        self._slots = [None] * world
        if errors:
            rank, err = errors[0]
            err.add_note(f"(raised on rank {rank} of {world})")
            raise err
        return results


def leftover_threads():
    return [t.name for t in threading.enumerate() if t.name.startswith(THREAD_PREFIX)]


@pytest.fixture
def thread_ranks(monkeypatch):
    """run(world, fn) with torch.distributed patched; afterwards no process group exists and no rank thread is alive"""
    ranks = InProcessRanks()
    ranks.install(monkeypatch)
    yield ranks.run
    monkeypatch.undo()
    assert not dist.is_initialized()
    assert not leftover_threads()
