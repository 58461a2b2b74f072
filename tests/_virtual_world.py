"""A world of G ranks as G threads of one process on one device: the multi-rank bodies of the sharded tests
(`body(rank, world, port, out, *args)`, written for one process per GPU) run unchanged at any G from 2 to 64.

`run_world(G, body, *args)` starts G threads; thread r is rank r.  While it runs, `torch.distributed`'s
is_initialized / get_world_size / get_rank / get_backend / init_process_group / destroy_process_group / barrier /
all_gather / all_reduce / broadcast talk to a coordinator instead of a process group, `torch.cuda.set_device` is a
no-op (every rank uses the current device), and `PeerExchange._symmetric` hands out plain device buffers: each rank
allocates and zeroes its own, the ranks meet, and every rank gets the same rank-ordered address array.  The exchange
kernels reach their peers only through that array, so they cannot tell G buffers on one device from G devices.

* The handle's `barrier` has the symmetric-memory barrier's meaning -- all work queued on every rank's current stream
  before it finishes before any work queued after it on any rank's current stream -- built from events: each rank
  records one on its current stream, the ranks meet on the host, each current stream waits for every rank's event,
  and the ranks meet again.  Every wait is for an event already recorded and nothing polls a flag on the device, so a
  protocol bug shows up as wrong numbers or a host-side error, never as a device hang.  What this does not exercise
  is NVLink and the device-side barrier of symmetric memory; the multi-process tests remain the only check of those.
* Collectives run on the host, in rank order, fully synchronously: the caller's stream is synchronised before its
  tensor is deposited, results are copied on the caller's stream and synchronised again before the closing meeting,
  so no rank frees or overwrites a tensor another rank's stream is still reading.  all_reduce sums in rank order and
  is deterministic.
* Each rank runs on a stream of its own, so the ranks overlap on the device as they do across GPUs and a missing
  barrier is a race, not a serialisation; and with multithreaded backward off (thread-local), so autograd runs every
  rank's backward on that rank's thread instead of one device worker shared by all callers (the first rank to wait in
  a barrier inside a backward would block the others).
* Every host meeting is a barrier with a timeout (`_Meeting`).  A rank that raises, or that reaches
  destroy_process_group, aborts it, so the others get BrokenBarrierError instead of waiting.  Every buffer handed out
  stays alive until all threads have ended and the device is synchronised: other ranks' streams store into it.

Everything is restored when run_world returns (pytest.MonkeyPatch.context).  CUDA is used only when the tensors are
on a CUDA device, so the host logic runs on CPU tensors as well."""
import contextlib
import queue
import sys
import threading
import time
import traceback

import pytest
import torch
import torch.distributed as dist

DEFAULT_TIMEOUT = 300.0


def _is_cuda(t):
    return isinstance(t, torch.Tensor) and t.is_cuda


class _Meeting:
    """A reusable host barrier of n threads with a timeout, like threading.Barrier, except that abort() breaks only
    the meetings not yet complete.  (threading.Barrier.abort also breaks the threads that the last arrival has released
    but that have not woken yet: a rank that passed the last meeting and leaves would fail the others.)"""

    def __init__(self, n, timeout):
        self.n, self.timeout = n, timeout
        self.cond = threading.Condition()
        self.count = self.generation = 0
        self.broken = False

    def wait(self):
        with self.cond:
            if self.broken:
                raise threading.BrokenBarrierError
            gen = self.generation
            self.count += 1
            if self.count == self.n:
                self.count, self.generation = 0, gen + 1
                self.cond.notify_all()
                return
            self.cond.wait_for(lambda: self.generation != gen or self.broken, self.timeout)
            if self.generation != gen:
                return
            self.broken = True                      # timed out or aborted: nobody waits here any more
            self.cond.notify_all()
            raise threading.BrokenBarrierError

    def abort(self):
        with self.cond:
            self.broken = True
            self.cond.notify_all()


class _World:
    """The coordinator: which thread is which rank, the host meetings, the buffers to keep alive."""

    def __init__(self, G, timeout):
        self.G, self.timeout = int(G), float(timeout)
        self.meeting = _Meeting(self.G, self.timeout)
        self.slots = [None] * self.G
        self.tls = threading.local()
        self.keep = []
        self.lock = threading.Lock()

    @property
    def rank(self):
        r = getattr(self.tls, "rank", None)
        if r is None:
            raise RuntimeError("virtual world: called from a thread that is not one of its ranks")
        return r

    def meet(self):
        self.meeting.wait()

    def abort(self):
        self.meeting.abort()

    def exchange(self, obj, between=None):
        """Deposit obj, meet, read every rank's (rank order), run between(objs) while no rank can move on, meet."""
        self.slots[self.rank] = obj
        self.meet()
        objs = list(self.slots)
        res = between(objs) if between is not None else None
        self.meet()
        return objs, res

    def hold(self, t):
        with self.lock:
            self.keep.append(t)


def _sync(t):
    if _is_cuda(t):
        torch.cuda.current_stream(t.device).synchronize()


class _Handle:
    """Stands in for the symmetric-memory handle: `buffer_ptrs` and an event-built `barrier`."""

    def __init__(self, world, ptrs):
        self.world, self.buffer_ptrs = world, list(ptrs)

    def barrier(self, channel=0, timeout_ms=0):
        w = self.world
        ev = None
        if torch.cuda.is_available():
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
        evs, _ = w.exchange(ev)
        if ev is not None:
            st = torch.cuda.current_stream()
            for e in evs:
                st.wait_event(e)


def peer_exchange_class():
    """The PeerExchange the layers use: the class of the module they live in ("dir_b200.sharded" imported by name
    would be a second copy of that module)."""
    import dir_b200
    return sys.modules[dir_b200.ShardedEmbeddingFM.__module__].PeerExchange


def _patch(mp, w):
    def _no_async(async_op):
        if async_op:
            raise NotImplementedError("virtual world: collectives are synchronous")

    def init_process_group(*a, rank=None, world_size=None, **kw):
        if rank is not None and rank != w.rank or world_size is not None and world_size != w.G:
            raise ValueError("virtual world: init_process_group(rank=%r, world_size=%r) on rank %d of %d"
                             % (rank, world_size, w.rank, w.G))

    def destroy_process_group(group=None):
        w.abort()               # the ranks still waiting would wait forever; a rank that is done needs no meeting

    def barrier(group=None, async_op=False, device_ids=None):
        _no_async(async_op)
        if torch.cuda.is_available():
            torch.cuda.current_stream().synchronize()
        w.meet()

    def all_gather(tensor_list, tensor, group=None, async_op=False):
        _no_async(async_op)
        if len(tensor_list) != w.G:
            raise ValueError("all_gather: tensor_list needs world_size entries")
        _sync(tensor)

        def copy(parts):
            for dst, src in zip(tensor_list, parts):
                dst.copy_(src)
            _sync(tensor_list[0])
        w.exchange(tensor, copy)

    def all_reduce(tensor, op=dist.ReduceOp.SUM, group=None, async_op=False):
        _no_async(async_op)
        if op != dist.ReduceOp.SUM:
            raise NotImplementedError("virtual world: all_reduce sums only")
        _sync(tensor)

        def total(parts):
            acc = parts[0].clone()
            for t in parts[1:]:
                acc.add_(t)
            _sync(acc)
            return acc
        _, acc = w.exchange(tensor, total)
        tensor.copy_(acc)       # after the closing meeting: nobody reads this rank's tensor any more
        _sync(tensor)

    def broadcast(tensor, src=None, group=None, async_op=False, group_src=None):
        _no_async(async_op)
        src = group_src if src is None else src
        if src is None or not 0 <= src < w.G:
            raise ValueError("broadcast: need 0 <= src < world_size")
        _sync(tensor)

        def take(parts):
            if w.rank != src:
                tensor.copy_(parts[src])
                _sync(tensor)
        w.exchange(tensor, take)

    def symmetric(group, world, n, dtype, device):
        if world != w.G:
            raise ValueError("virtual world: PeerExchange for %d ranks in a world of %d" % (world, w.G))
        buf = torch.zeros(n, dtype=dtype, device=device)
        _sync(buf)                                  # zeroed before any peer can store into it
        w.hold(buf)
        ptrs, _ = w.exchange(buf.data_ptr())
        return buf, _Handle(w, ptrs), torch.tensor(ptrs, dtype=torch.int64, device=device)

    PeerExchange = peer_exchange_class()
    for name, fn in (("is_initialized", lambda: True), ("get_world_size", lambda group=None: w.G),
                     ("get_rank", lambda group=None: w.rank), ("get_backend", lambda group=None: "nccl"),
                     ("init_process_group", init_process_group), ("destroy_process_group", destroy_process_group),
                     ("barrier", barrier), ("all_gather", all_gather), ("all_reduce", all_reduce),
                     ("broadcast", broadcast)):
        mp.setattr(dist, name, fn)
    mp.setattr(torch.cuda, "set_device", lambda device: None)
    mp.setattr(PeerExchange, "_symmetric", staticmethod(symmetric))
    mp.setenv("MASTER_ADDR", "127.0.0.1")          # (the bodies set them for a real rendezvous; restored afterwards)
    mp.setenv("MASTER_PORT", "0")


def run_world(G, body, *args, timeout=DEFAULT_TIMEOUT):
    """Run body(rank, G, port, out, *args) on G threads, each on a CUDA stream of its own when CUDA is available ->
    what the ranks put into `out`, sorted by rank.  Raises if a rank raised out of its body or did not finish in time."""
    w = _World(G, timeout)
    out = queue.Queue()
    errors = [None] * w.G
    cuda = torch.cuda.is_available()

    def main(r):
        w.tls.rank = r
        try:
            with contextlib.ExitStack() as es:
                es.enter_context(torch.autograd.set_multithreading_enabled(False))
                if cuda:
                    s = torch.cuda.Stream()
                    es.enter_context(torch.cuda.stream(s))
                body(r, w.G, 0, out, *args)
                if cuda:
                    s.synchronize()
        except BaseException:
            errors[r] = traceback.format_exc()
            w.abort()

    with pytest.MonkeyPatch.context() as mp:
        _patch(mp, w)
        threads = [threading.Thread(target=main, args=(r,), name="rank%d" % r, daemon=True) for r in range(w.G)]
        for t in threads:
            t.start()
        deadline = time.monotonic() + w.timeout + 60.0
        for t in threads:
            t.join(max(0.0, deadline - time.monotonic()))
        late = [r for r, t in enumerate(threads) if t.is_alive()]
        if late:
            w.abort()
            for t in threads:
                t.join(30.0)
        if cuda:
            torch.cuda.synchronize()
    w.keep.clear()
    if late:
        raise RuntimeError("virtual world of %d: ranks %s did not finish within %.0f s" % (w.G, late, w.timeout))
    failed = [(r, e) for r, e in enumerate(errors) if e is not None]
    if failed:
        raise AssertionError("virtual world of %d: %s" % (w.G, "\n".join("rank %d:\n%s" % f for f in failed)))
    res = []
    while not out.empty():
        res.append(out.get())
    return sorted(res, key=lambda x: x[0])
