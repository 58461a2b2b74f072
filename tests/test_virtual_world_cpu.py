"""The host logic of tests/_virtual_world.py on CPU tensors: the rendezvous of the exchange buffers, the collectives,
the thread-local rank, failing fast when a rank raises, and torch.distributed restored afterwards.  (The device part
-- streams, events -- runs in tests/test_gpu_sharded_virtual.py.)"""
import threading
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist

from tests._virtual_world import peer_exchange_class, run_world

SIZES = [1, 2, 3, 8]


def _body(fn):
    """A rank body that reports fn(rank, world) or the traceback, as the multi-rank bodies do."""
    def body(rank, world, port, out):
        dist.init_process_group("nccl", rank=rank, world_size=world)
        try:
            out.put((rank, fn(rank, world)))
        except Exception:
            import traceback
            out.put((rank, traceback.format_exc()))
        finally:
            dist.destroy_process_group()
    return body


def _values(rank, shape=(5, 3), dtype=torch.float32):
    """Per-rank values whose float sums round differently in different orders."""
    g = torch.Generator().manual_seed(100 + rank)
    return (torch.randn(shape, generator=g, dtype=torch.float64) * 10.0 ** (rank % 5)).to(dtype)


@pytest.mark.parametrize("G", SIZES)
def test_rank_world_and_backend(G):
    def fn(rank, world):
        torch.cuda.set_device(rank)                     # a no-op: every rank uses one device
        return (dist.is_initialized(), dist.get_world_size(), dist.get_rank(), dist.get_backend(),
                threading.current_thread().name)
    res = run_world(G, _body(fn))
    assert res == [(r, (True, G, r, "nccl", "rank%d" % r)) for r in range(G)]


@pytest.mark.parametrize("G", SIZES)
def test_rendezvous_hands_out_rank_ordered_addresses(G):
    PeerExchange = peer_exchange_class()

    def fn(rank, world):
        bufs = []
        for n, dtype in ((1000 + rank, torch.uint8), (7, torch.float64)):     # two rendezvous in a row
            buf, h, base = PeerExchange._symmetric(None, world, n, dtype, "cpu")
            assert buf.numel() == n and buf.dtype == dtype and not bool(buf.any()), "zeroed, own size"
            assert base.dtype == torch.int64 and base.tolist() == h.buffer_ptrs
            assert h.buffer_ptrs[rank] == buf.data_ptr()
            h.barrier(channel=0, timeout_ms=1000)
            bufs.append(buf)
        return [b.data_ptr() for b in bufs], h.buffer_ptrs
    res = run_world(G, _body(fn))
    assert [r for r, _ in res] == list(range(G)) and not any(isinstance(v, str) for _, v in res), res
    mine = [v[0] for _, v in res]
    # every rank got the same array: the second buffers of ranks 0 .. G-1, in rank order
    assert all(v[1] == [m[1] for m in mine] for _, v in res)
    assert len(set(m[0] for m in mine)) == G


@pytest.mark.parametrize("G", SIZES)
def test_collectives(G):
    def fn(rank, world):
        x = _values(rank)
        parts = [torch.full((5, 3), -1.0) for _ in range(world)]
        dist.all_gather(parts, x)
        s = x.clone()
        dist.all_reduce(s)
        i = torch.tensor([rank + 1, 10 * rank], dtype=torch.int64)
        dist.all_reduce(i)
        b = x.clone()
        dist.broadcast(b, world - 1)
        dist.barrier()
        assert torch.equal(x, _values(rank)), "the collectives leave the input alone"
        return [p.numpy() for p in parts], s.numpy(), i.tolist(), b.numpy()
    res = run_world(G, _body(fn))
    want = [_values(r).numpy() for r in range(G)]
    total = want[0].copy()
    for w in want[1:]:
        total = total + w                               # float32, rank order
    for r, (parts, s, i, b) in res:
        assert all(np.array_equal(p, w) for p, w in zip(parts, want))
        assert s.tobytes() == total.tobytes(), "all_reduce: the rank-order float32 sum, bit for bit"
        assert i == [G * (G + 1) // 2, 10 * G * (G - 1) // 2]
        assert np.array_equal(b, want[G - 1])
    if G >= 3:      # the order matters for these values: a sum in another order would be caught
        other = want[G - 1].copy()
        for w in want[G - 2::-1]:
            other = other + w
        assert other.tobytes() != total.tobytes()


def test_a_rank_that_raises_fails_the_others_fast():
    """Rank 1 raises before a collective the other ranks wait in: they get BrokenBarrierError long before the
    meeting's timeout, and run_world reports every rank."""
    def body(rank, world, port, out):
        if rank == 1:
            raise ValueError("rank 1 fails")
        x = torch.ones(2)
        dist.all_reduce(x)
        out.put((rank, "ok"))
    start = time.monotonic()
    with pytest.raises(AssertionError) as ei:
        run_world(4, body, timeout=120.0)
    assert time.monotonic() - start < 30.0, "the other ranks must not wait for the timeout"
    msg = str(ei.value)
    assert "rank 1 fails" in msg and "BrokenBarrierError" in msg
    assert all("rank %d:" % r in msg for r in range(4))


def test_a_rank_that_reports_and_leaves_fails_the_others_fast():
    """The multi-rank bodies catch their own exceptions, report them and call destroy_process_group: a rank that
    leaves early aborts the meetings the others are waiting in."""
    def fn(rank, world):
        if rank == 0:
            raise AssertionError("rank 0 disagrees")
        x = torch.ones(1)
        dist.all_reduce(x)
        return "ok"
    res = run_world(3, _body(fn), timeout=120.0)
    assert "rank 0 disagrees" in res[0][1]
    assert all("BrokenBarrierError" in v for _, v in res[1:])


def test_a_rank_that_never_arrives_times_out():
    def body(rank, world, port, out):
        if rank == 0:
            dist.barrier()
        out.put((rank, "ok"))
    with pytest.raises(AssertionError) as ei:
        run_world(2, body, timeout=1.0)
    assert "BrokenBarrierError" in str(ei.value)


def test_torch_distributed_is_restored():
    PeerExchange = peer_exchange_class()
    names = ("is_initialized", "get_world_size", "get_rank", "get_backend", "init_process_group",
             "destroy_process_group", "barrier", "all_gather", "all_reduce", "broadcast")
    before = {n: getattr(dist, n) for n in names}
    sym, set_device = PeerExchange.__dict__["_symmetric"], torch.cuda.set_device
    seen = run_world(2, _body(lambda rank, world: dist.get_world_size is before["get_world_size"]))
    assert seen == [(0, False), (1, False)]
    assert all(getattr(dist, n) is f for n, f in before.items())
    assert PeerExchange.__dict__["_symmetric"] is sym and torch.cuda.set_device is set_device
    assert not dist.is_initialized()
