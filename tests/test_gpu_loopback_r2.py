"""R2 (compiled-graph communicator + TorchTensor channel) and N1 (RDT transport) on ONE GPU.

Same checks as tests/test_gpu_communicator.py and tests/test_gpu_rdt.py — which need one process per
GPU — but with every endpoint of the group living in a thread of this process on cuda:0 (its own
CUDA stream, its own B200Communicator, a shared in-memory rendezvous store), so a single-GPU box
exercises the real communicator, channel, header ring, multi-reader ring and RDT code down to the
kernels.  Follows the reference's GPU DAG tests (python/ray/dag/tests/experimental/
test_torch_tensor_dag.py): p2p with varying shapes (:213-268), dedicated communication streams
(:373-415), collectives for every reduce op compared with torch.equal against
torch.sum/prod/min/max of the stacked inputs (:1340-1450), wrong-shape allreduce surfaces
RayChannelError instead of hanging (:1544-1588), destroyed group raises RayChannelError, and a custom
communicator class picked through the accelerator-context registry (:472-571,
accelerator_context.py:222-233).
"""
import os
import queue
import threading

import pytest
import torch

from ant_ray_b200 import _native as N

pytestmark = pytest.mark.gpu


class Endpoints:
    """W B200Communicator endpoints on cuda:0, one thread each."""

    def __init__(self, world, overlap=False, blocking_errors=None, comm_id=None, timeout_ms=15000, cls=None):
        from ant_ray_b200.b200_group import make_config
        from ant_ray_b200.communicator import B200Communicator
        from ant_ray_b200.loopback import _MemStore

        self.world = world
        store = _MemStore()
        comm_id = comm_id or B200Communicator.generate_communicator_id()
        sm = torch.cuda.get_device_properties(0).multi_processor_count
        cfg = dict(max_blocks=max(1, (2 * sm) // world - 2), staging_bytes=8 << 20, timeout_ms=timeout_ms)
        self.streams = [torch.cuda.Stream(device=0) for _ in range(world)]
        self.comms = [None] * world
        prev = os.environ.get("B200COLL_MULTICAST")
        os.environ["B200COLL_MULTICAST"] = "0"  # one device cannot join a multicast object twice
        try:
            def make(r):
                torch.cuda.set_device(0)
                kw = {} if blocking_errors is None else {"blocking_errors": blocking_errors}
                self.comms[r] = (cls or B200Communicator)(world, comm_id, r, list(range(world)), self.streams[r], overlap,
                                                          store=store, config=make_config(**cfg), **kw)
            self.run(make)
        finally:
            if prev is None:
                os.environ.pop("B200COLL_MULTICAST", None)
            else:
                os.environ["B200COLL_MULTICAST"] = prev

    def run(self, fn, ranks=None):
        """fn(rank) in one thread per rank, under that rank's stream; returns the results by rank."""
        ranks = list(range(self.world)) if ranks is None else list(ranks)
        out, errs = {}, {}

        def body(r):
            try:
                torch.cuda.set_device(0)
                with torch.cuda.stream(self.streams[r]):
                    out[r] = fn(r)
                    self.streams[r].synchronize()
            except BaseException as e:  # noqa: BLE001
                errs[r] = e

        ts = [threading.Thread(target=body, args=(r,)) for r in ranks]
        for t in ts:
            t.start()
        for t in ts:
            t.join(120)
        assert not any(t.is_alive() for t in ts), "an endpoint thread is stuck"
        if errs:
            raise next(iter(errs.values()))
        return [out[r] for r in ranks]

    def close(self):
        for c in self.comms:
            if c is not None:
                c.destroy()


class QueueMeta:
    """Metadata side channel for endpoints that do not inline headers: one queue per reader."""

    def __init__(self, readers):
        self.q = {r: queue.Queue() for r in readers}
        self.writes = 0
        self.reads = 0

    def for_rank(self, rank):
        outer = self

        class View:
            def write(self, obj, timeout=None):
                outer.writes += 1
                for q in outer.q.values():
                    q.put(obj)

            def read(self, timeout=None):
                outer.reads += 1
                return outer.q[rank].get(timeout=timeout or 30)

            def close(self):
                pass

        return View()


@pytest.fixture
def pair():
    made = []

    def make(world=2, **kw):
        e = Endpoints(world, **kw)
        made.append(e)
        return e

    yield make
    for e in made:
        e.close()


@pytest.mark.parametrize("overlap", [False, True])
@pytest.mark.parametrize("inline", [True, False])
def test_p2p_varying_shapes(pair, overlap, inline):
    """Dynamic shapes: every message announces (shape, dtype) — through the header ring when inlined (no
    metadata channel traffic at all), through the side channel otherwise."""
    from ant_ray_b200.channel import TensorListChannel

    e = pair(2, overlap=overlap)
    meta = QueueMeta([1])
    chans = [TensorListChannel(e.comms[r], 0, [1], meta.for_rank(r), inline_metadata=inline) for r in range(2)]
    for i, shape in enumerate([(10,), (20, 3), (1,), (4, 5, 6), (0,), (100_000,)]):
        ts = [torch.full(shape, float(i), dtype=torch.float16, device="cuda"), torch.full((3,), i + 1, dtype=torch.int64, device="cuda")]

        def step(r):
            if r == 0:
                with e.comms[0].send_stream:
                    chans[0].write(ts)
                return None
            with e.comms[1].recv_stream:
                got = chans[1].read(timeout=30)
            torch.cuda.synchronize()
            return [g.cpu() for g in got]

        got = e.run(step)[1]
        assert torch.equal(got[0], torch.full(shape, float(i), dtype=torch.float16)) and got[0].shape == torch.Size(shape)
        assert torch.equal(got[1], torch.full((3,), i + 1, dtype=torch.int64))
    assert (meta.writes, meta.reads) == ((0, 0) if inline else (6, 6))
    for c in e.comms:
        c.check()


def test_static_shape_sends_metadata_once_and_empty_lists(pair):
    from ant_ray_b200.channel import TensorListChannel

    e = pair(2)
    meta = QueueMeta([1])
    chans = [TensorListChannel(e.comms[r], 0, [1], meta.for_rank(r), static_shape=True) for r in range(2)]
    for i in range(4):
        t = torch.full((50_000,), float(i), dtype=torch.float16, device="cuda")
        got = e.run(lambda r: chans[0].write([t]) if r == 0 else [x.cpu() for x in chans[1].read(30)])[1]
        assert (got[0] == i).all()
    hdr_out = e.comms[0]._hdr_out[(0, 1)]
    assert hdr_out.count == 1, "static shape: only the first message carries a header"
    with pytest.raises(ValueError):
        chans[0].write([torch.ones(3, device="cuda")])  # shape changed under static_shape
    # an empty tensor list is a message too (header with count 0, no payload)
    chans2 = [TensorListChannel(e.comms[r], 1, [0], meta.for_rank(r)) for r in range(2)]
    got = e.run(lambda r: chans2[1].write([]) if r == 1 else chans2[0].read(30))[0]
    assert got == []


def test_value_channel_with_cpu_remainder_and_direct_return(pair):
    from ant_ray_b200.channel import TensorListChannel, TorchTensorChannel

    e = pair(2)
    meta, cpu = QueueMeta([1]), QueueMeta([1])
    chans = [TorchTensorChannel(TensorListChannel(e.comms[r], 0, [1], meta.for_rank(r)), cpu.for_rank(r)) for r in range(2)]
    value = {"t": torch.arange(12, device="cuda").reshape(3, 4), "tag": "hello", "n": 3, "u": torch.ones(5, device="cuda") * 7}
    got = e.run(lambda r: chans[0].write(value) if r == 0 else chans[1].read(30))[1]
    assert torch.equal(got["t"].cpu(), torch.arange(12).reshape(3, 4)) and got["tag"] == "hello" and got["n"] == 3
    assert torch.equal(got["u"].cpu(), torch.ones(5) * 7)
    direct = [TorchTensorChannel(TensorListChannel(e.comms[r], 1, [0], meta.for_rank(r)), cpu.for_rank(r), direct_return=True) for r in range(2)]
    got = e.run(lambda r: direct[1].write(torch.ones(9, device="cuda") * 3) if r == 1 else direct[0].read(30))[0]
    assert torch.equal(got.cpu(), torch.ones(9) * 3)
    with pytest.raises(ValueError):
        direct[1].write({"not": "a tensor"})


@pytest.mark.parametrize("world", [3, 4])
def test_multi_reader_channel_sends_once(pair, world):
    """N2: one writer, several readers: each tensor leaves the writer in ONE send (the multi-reader ring;
    a multicast store stream on a multi-GPU box, unicast stores here), not once per reader
    (reference :586-590 TODO)."""
    from ant_ray_b200.channel import TensorListChannel

    e = pair(world)
    readers = list(range(1, world))
    chans = [TensorListChannel(e.comms[r], 0, readers, QueueMeta(readers).for_rank(r)) for r in range(world)]
    launches0 = N.launch_count()
    n_msgs = 5
    for i in range(n_msgs):
        # 100 messages would wrap the 64-cell ring many times; sizes straddle the 32 KiB cell
        ts = [torch.full((70_000 + i,), float(i), dtype=torch.float32, device="cuda"), torch.arange(5 + i, device="cuda")]

        def step(r):
            if r == 0:
                chans[0].write(ts)
                return None
            return [g.cpu() for g in chans[r].read(30)]

        res = e.run(step)
        for r in readers:
            assert torch.equal(res[r][0], torch.full((70_000 + i,), float(i))) and torch.equal(res[r][1], torch.arange(5 + i))
    # 2 tensors per message: 1 send_multi + (world-1) recvs each
    assert N.launch_count() - launches0 == n_msgs * 2 * (1 + len(readers))
    # ring wrap: a message of 3 x 64 cells goes through the 64-cell multi-reader ring with per-reader acks
    big = torch.randint(0, 255, (3 * 64 * (32 << 10) + 17,), dtype=torch.uint8, device="cuda")
    res = e.run(lambda r: chans[0].write([big]) if r == 0 else chans[r].read(30)[0].cpu())
    for r in readers:
        assert torch.equal(res[r], big.cpu())
    # a second reader set from the same writer is refused by the native layer, and served by per-reader sends
    other = [TensorListChannel(e.comms[r], 0, [1], QueueMeta([1]).for_rank(r)) for r in range(2)]
    got = e.run(lambda r: other[0].write([torch.ones(4, device="cuda")]) if r == 0 else other[1].read(30)[0].cpu(), ranks=[0, 1])[1]
    assert torch.equal(got, torch.ones(4))
    if world > 3:
        bad = TensorListChannel(e.comms[0], 0, [1, 2], QueueMeta([1, 2]).for_rank(0))
        from ant_ray_b200.communicator import RayChannelError
        with pytest.raises(RayChannelError):
            bad.write([torch.ones(4, device="cuda")])
    for c in e.comms:
        c.check()


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_collectives_match_torch(pair, world, dtype):
    from ant_ray_b200.types import DagReduceOp

    e = pair(world)
    n = world * 3000
    ins = [torch.randn(n, generator=torch.Generator().manual_seed(100 + r)).to(dtype) for r in range(world)]
    stacked = torch.stack(ins)
    # The ranks are threads of one process, so a device allocation made by one rank while another rank's kernel
    # already waits for it can itself wait for that kernel.  Every buffer is therefore allocated in a round of its
    # own before the collective is issued; outputs start as NaN so that an element the kernel did not write fails.
    xs = e.run(lambda r: ins[r].cuda())

    def collective(out_numel, fn):
        outs = e.run(lambda r: torch.full((out_numel,), float("nan"), dtype=dtype, device="cuda"))
        e.run(lambda r: fn(r, xs[r], outs[r]))
        for c in e.comms:
            c.check()
        return [o.cpu() for o in outs]

    expect = {"MIN": stacked.min(0).values, "MAX": stacked.max(0).values}
    if world == 2:  # order-independent: exact (test_torch_tensor_dag.py:1340-1450)
        expect.update({"SUM": stacked.sum(0), "PRODUCT": stacked.prod(0), "AVG": (stacked.float().sum(0) / 2).to(dtype)})
    for op, want in expect.items():
        for o in collective(n, lambda r, x, out: e.comms[r].allreduce(x, out, getattr(DagReduceOp, op))):
            assert torch.equal(o, want), op
    if world > 2:  # the kernels fold ranks 0..W-1 in order with fp32 accumulation: compare with exactly that
        from oracle import oracle as O
        for o in collective(n, lambda r, x, out: e.comms[r].allreduce(x, out, DagReduceOp.SUM)):
            assert torch.equal(o, O.allreduce(ins))

    for o in collective(n * world, lambda r, x, out: e.comms[r].allgather(x, out)):
        assert torch.equal(o, torch.cat(ins))

    for r, o in enumerate(collective(n // world, lambda r, x, out: e.comms[r].reducescatter(x, out, DagReduceOp.MAX))):
        assert torch.equal(o, stacked.max(0).values[r * (n // world):(r + 1) * (n // world)])


@pytest.mark.parametrize("blocking", [True, False])
def test_wrong_shape_raises_channel_error_not_hang(pair, blocking):
    """Blocking errors: the failing call raises (reference behaviour).  Deferred (default, N4): the call
    returns after enqueue and the error is raised by check() / the next call."""
    from ant_ray_b200.communicator import RayChannelError

    e = pair(2, blocking_errors=blocking, timeout_ms=5000)

    def step(r):
        x = torch.ones(100_000 * (r + 1), device="cuda")   # beyond the LL range: both ranks see the mismatch in the flag round
        try:
            e.comms[r].allreduce(x, torch.empty_like(x))
        except RayChannelError as err:
            return "call: " + str(err)[:40]
        try:
            e.comms[r].check()
        except RayChannelError as err:
            return "check: " + str(err)[:40]
        return "no error"

    res = e.run(step)
    assert all(x.startswith("call" if blocking else "check") for x in res), res
    # poisoned: the next call raises immediately in both modes
    with pytest.raises(RayChannelError):
        e.comms[0].send(torch.ones(4, device="cuda"), 1)


def test_recv_does_not_block_the_host(pair):
    """N4: recv returns once the kernel is enqueued (nccl_group.py:215,237 'TODO: Avoid CUDA
    synchronization'): the receiver can return from recv before the sender has even started."""
    e = pair(2, timeout_ms=20000)
    alloc = lambda shape, dtype: torch.empty(shape, dtype=dtype, device="cuda")  # noqa: E731
    returned = threading.Event()
    res = {}

    def receiver():
        torch.cuda.set_device(0)
        with torch.cuda.stream(e.streams[1]):
            buf = e.comms[1].recv((1 << 16,), torch.float32, 0, alloc)
            returned.set()           # no sender yet: the host was not blocked
            y = buf * 2               # consumer work enqueued behind the receive on the same stream
            e.streams[1].synchronize()
            res["y"] = y.cpu()

    t = threading.Thread(target=receiver)
    t.start()
    assert returned.wait(10), "recv blocked the host although nothing had been sent"
    with torch.cuda.stream(e.streams[0]):
        e.comms[0].send(torch.full((1 << 16,), 21.0, device="cuda"), 1)
    t.join(30)
    assert not t.is_alive() and bool((res["y"] == 42).all())
    e.comms[1].check()


def test_destroy_raises_channel_error(pair):
    from ant_ray_b200.communicator import RayChannelError

    e = pair(2)
    e.comms[0].destroy()
    with pytest.raises(RayChannelError):
        e.comms[0].send(torch.ones(4, device="cuda"), 1)
    with pytest.raises(RayChannelError):
        e.comms[0].recv((4,), torch.float32, 1, lambda s, d: torch.empty(s, dtype=d, device="cuda"))
    with pytest.raises(RayChannelError):
        e.comms[0].check()


def test_microbenchmark_shape_100kB_fp16(pair):
    """compiled_graph_gpu_microbenchmark.py:441-451: 100,000-byte fp16 tensor, sender -> receiver."""
    import time

    e = pair(2)
    n, iters = 50_000, 200
    t = torch.ones(n, dtype=torch.float16, device="cuda")
    alloc = lambda shape, dtype: torch.empty(shape, dtype=dtype, device="cuda")  # noqa: E731

    def step(r):
        t0 = time.perf_counter()
        for _ in range(iters):
            if r == 0:
                e.comms[0].send(t, 1)
            else:
                e.comms[1].recv((n,), torch.float16, 0, alloc)
        torch.cuda.current_stream().synchronize()
        return (time.perf_counter() - t0) / iters * 1e6

    us = e.run(step)
    print(f"loopback p2p 100kB fp16: sender {us[0]:.1f} us/msg, receiver {us[1]:.1f} us/msg")
    assert us[1] < 2000


def test_accelerator_context_registry_builds_the_communicator(pair):
    """a18: `register_accelerator_context("cuda", B200Communicator)` makes the driver-orchestrated
    _do_init_communicator build a B200Communicator with the registry's own positional call
    (torch_tensor_accelerator_channel.py:673-680), with real handles as `actor_handles`."""
    from ant_ray_b200 import accelerator_context as AC
    from ant_ray_b200 import channel_context as CC
    from ant_ray_b200.communicator import B200Communicator
    from ant_ray_b200.loopback import _MemStore

    store = _MemStore()
    made = []

    class Registered(B200Communicator):
        """What a deployment registers; here it also injects the in-process rendezvous store."""

        def __init__(self, world_size, comm_id, rank, actor_handles, cuda_stream, use_communication_streams=False):
            from ant_ray_b200.b200_group import make_config

            super().__init__(world_size, comm_id, rank, actor_handles, cuda_stream, use_communication_streams, store=store,
                             config=make_config(max_blocks=64, staging_bytes=4 << 20, timeout_ms=15000))
            made.append(self)

    class Handle:  # stands in for an ActorHandle: identity is what get_rank() uses
        def __init__(self, i):
            self._ray_actor_id = f"actor-{i}"

    handles = [Handle(0), Handle(1)]
    AC.register_accelerator_context("cuda", Registered)
    prev = os.environ.get("B200COLL_MULTICAST")
    os.environ["B200COLL_MULTICAST"] = "0"
    try:
        assert AC.is_accelerator_context_registered() and AC.AcceleratorContext.get().communicator_cls is Registered
        comm_id = CC._do_get_unique_communication_id(None)
        ctxs = [CC.ChannelContext() for _ in range(2)]
        streams = [torch.cuda.Stream() for _ in range(2)]

        def init(r):
            torch.cuda.set_device(0)
            with torch.cuda.stream(streams[r]):
                # one ChannelContext per "actor": each thread plays one actor process
                CC.ChannelContext._current = None
                c = AC.AcceleratorContext.get().create_communicator(2, comm_id, r, handles, torch.cuda.current_stream(), False)
                ctxs[r].communicators["g"] = c

        ts = [threading.Thread(target=init, args=(r,)) for r in range(2)]
        [t.start() for t in ts]
        [t.join(60) for t in ts]
        c0, c1 = ctxs[0].communicators["g"], ctxs[1].communicators["g"]
        assert isinstance(c0, Registered) and c0.get_world_size() == 2 and c0.get_transport_name() == "accelerator"
        assert c0.get_rank(handles[1]) == 1 and c1.get_self_rank() == 1 and c0.get_actor_handles() is handles
        with pytest.raises(ValueError):
            c0.get_rank(Handle(7))
        x = torch.arange(1000, dtype=torch.float32, device="cuda")
        got = {}

        def go(r):
            torch.cuda.set_device(0)
            with torch.cuda.stream(streams[r]):
                if r == 0:
                    c0.send(x, 1)
                else:
                    got["y"] = c1.recv((1000,), torch.float32, 0, lambda s, d: torch.empty(s, dtype=d, device="cuda"))
                streams[r].synchronize()

        ts = [threading.Thread(target=go, args=(r,)) for r in range(2)]
        [t.start() for t in ts]
        [t.join(60) for t in ts]
        assert torch.equal(got["y"].cpu(), x.cpu())
    finally:
        AC.AcceleratorContext.set(None)
        if prev is None:
            os.environ.pop("B200COLL_MULTICAST", None)
        else:
            os.environ["B200COLL_MULTICAST"] = prev
        for c in made:
            c.destroy()


def test_rdt_transport_loopback():
    """N1: RDT tensor transport -> ray.util.collective send/recv -> B200Group -> kernels, both ranks in
    this process (each rank's group registered under its own name, sharing one rendezvous key)."""
    from ant_ray_b200 import collective as col
    from ant_ray_b200.b200_group import B200Group, make_config
    from ant_ray_b200.loopback import _MemStore
    from ant_ray_b200.rdt_transport import B200TensorTransport, CollectiveCommunicatorMetadata

    store = _MemStore()
    cfg = dict(max_blocks=64, staging_bytes=4 << 20, timeout_ms=15000)
    names = ["rdt-lb/rank0", "rdt-lb/rank1"]
    prev = os.environ.get("B200COLL_MULTICAST")
    os.environ["B200COLL_MULTICAST"] = "0"
    try:
        for r, name in enumerate(names):
            g = B200Group(2, r, name, store=store, device=0, config=make_config(**cfg))
            g._key = "b200coll/rdt-lb"   # one group seen from two "actors"
            col._group_mgr._name_group_map[name] = g
        tt = B200TensorTransport()
        assert tt.tensor_transport_backend == "B200" and not tt.is_one_sided() and not tt.can_abort_transport()
        payload = [torch.arange(12, dtype=torch.float32, device="cuda").reshape(3, 4), torch.full((100_000,), 3, dtype=torch.bfloat16, device="cuda")]
        tmeta = tt.extract_tensor_transport_metadata("obj", payload)
        assert [tuple(s) for s, _ in tmeta.tensor_meta] == [(3, 4), (100_000,)] and tmeta.tensor_device.type == "cuda"
        bufs = [torch.empty(tuple(s), dtype=d, device="cuda") for s, d in tmeta.tensor_meta]
        streams = [torch.cuda.Stream(), torch.cuda.Stream()]
        errs = []

        def side(r):
            try:
                torch.cuda.set_device(0)
                with torch.cuda.stream(streams[r]):
                    if r == 0:
                        tt.send_multiple_tensors(payload, tmeta, CollectiveCommunicatorMetadata(names[0], 0, 1))
                    else:
                        tt.recv_multiple_tensors(bufs, "obj", tmeta, CollectiveCommunicatorMetadata(names[1], 0, 1))
                    streams[r].synchronize()
            except BaseException as e:  # noqa: BLE001
                errs.append(e)

        ts = [threading.Thread(target=side, args=(r,)) for r in range(2)]
        [t.start() for t in ts]
        [t.join(60) for t in ts]
        assert not errs, errs
        assert torch.equal(bufs[0].cpu(), payload[0].cpu()) and torch.equal(bufs[1].cpu(), payload[1].cpu())
        # a transfer that fails on the device raises from recv_multiple_tensors instead of returning garbage
        tt.abort_transport("obj", CollectiveCommunicatorMetadata(names[1], 0, 1))
        with pytest.raises(RuntimeError):
            with torch.cuda.stream(streams[1]):
                tt.recv_multiple_tensors(bufs[:1], "obj2", tmeta, CollectiveCommunicatorMetadata(names[1], 0, 1))
    finally:
        if prev is None:
            os.environ.pop("B200COLL_MULTICAST", None)
        else:
            os.environ["B200COLL_MULTICAST"] = prev
        for name in names:
            col._group_mgr.destroy_collective_group(name)
