"""Compiled-Graph boundary (B2): ``B200Communicator`` and the GPU tensor channel.

Mirrors the behavioural spec in python/ray/dag/tests/experimental/test_torch_tensor_dag.py
(p2p :100-250, static shape / direct return, custom communicator :469-601, collectives with
``torch.equal`` on randn fp16 :1348-1459, wrong shape) and test_cpu_communicator_dag.py.
Actors are threads here; every actor owns a communicator endpoint and CUDA streams.
"""
import pickle
import threading
import time

import numpy as np
import pytest
import torch

from oracle import collective_oracle as O

pytestmark = pytest.mark.gpu


class Actors:
    def __init__(self, n, **comm_kwargs):
        from ray_b200.channel import B200Communicator
        from ray_b200.store import DictStore

        self.n = n
        ndev = torch.cuda.device_count()
        self.devices = [r % ndev for r in range(n)] if ndev < n else list(range(n))
        self.shared = len(set(self.devices)) < n
        store = DictStore()
        handles = [f"actor-{i}" for i in range(n)]
        template = B200Communicator(n, actor_handles=handles, store=store, timeout_ms=15000,
                                    staging_bytes=8 << 20, inbox_bytes=2 << 20, **comm_kwargs)
        # the driver-side object knows ranks before initialize (test_torch_tensor_dag.py:500-514)
        assert template.get_world_size() == n and template.get_rank("actor-1") == 1
        assert template.get_self_rank() is None
        self.comms = []
        for r in range(n):
            c = B200Communicator(n, template._comm_id, None, handles, None,
                                 comm_kwargs.get("use_communication_streams", False), store, self.devices[r],
                                 timeout_ms=15000, staging_bytes=8 << 20, inbox_bytes=2 << 20)
            self.comms.append(c)
        # One persistent stream per actor, with a warmed-up caching-allocator pool.  When actors share
        # a GPU (fewer devices than ranks) this is a correctness matter for the HARNESS, not for the
        # library: CUDA forbids two kernels from running concurrently if a device (or pinned)
        # allocation is issued between their launches (implicit synchronisation), so a cudaMalloc
        # by one actor between another actor's launch and its own would serialise two kernels that
        # wait for each other.  Allocations served from torch's cache issue no CUDA call.  (In
        # production every rank owns its GPU and no co-dependent kernels share a device.)
        self.streams = [torch.cuda.Stream(self.devices[r]) for r in range(n)]
        for r in range(n):
            with torch.cuda.device(self.devices[r]), torch.cuda.stream(self.streams[r]):
                warm = [torch.empty(1 << 19, dtype=torch.uint8, device=self.dev(r)) for _ in range(3)]
                warm += [torch.empty(24 << 20, dtype=torch.uint8, device=self.dev(r))]
                del warm
        torch.cuda.synchronize()
        self.run(lambda r, c: c.initialize(r))
        if self.shared:
            for c in self.comms:
                c.comm.set_blocks(max(1, 140 // n))

    def run(self, fn):
        out, err = [None] * self.n, [None] * self.n

        def body(r):
            try:
                torch.cuda.default_stream(self.devices[r]).synchronize()
                with torch.cuda.device(self.devices[r]), torch.cuda.stream(self.streams[r]):
                    self.comms[r]._cuda_stream = self.comms[r]._cuda_stream or torch.cuda.current_stream()
                    out[r] = fn(r, self.comms[r])
                    torch.cuda.current_stream().synchronize()
            except BaseException as e:  # noqa: BLE001
                err[r] = e

        ts = [threading.Thread(target=body, args=(r,)) for r in range(self.n)]
        [t.start() for t in ts]
        [t.join(120) for t in ts]
        for e in err:
            if e is not None:
                raise e
        for c in self.comms:  # a kernel that gave up (watchdog) leaves its output unwritten
            if c.comm is not None and not c.comm.closed:
                c.comm.check_status()
        return out

    def dev(self, r):
        return torch.device("cuda", self.devices[r])

    def close(self):
        for c in self.comms:
            c.destroy()


@pytest.fixture()
def actors(native_lib):
    made = []

    def make(n, **kw):
        a = Actors(n, **kw)
        made.append(a)
        return a

    yield make
    for a in made:
        a.close()


def _alloc(dev):
    return lambda shape, dtype: torch.empty(shape, dtype=dtype, device=dev)


def test_communicator_contract_and_pickling(actors):
    from ray_b200.channel import B200Communicator

    a = actors(2)
    c = a.comms[0]
    assert c.get_transport_name() == "accelerator"
    assert c.get_self_rank() == 0 and a.comms[1].get_self_rank() == 1
    assert c.get_actor_handles() == ["actor-0", "actor-1"]
    with pytest.raises(ValueError):
        c.get_rank("stranger")
    assert isinstance(B200Communicator.generate_communicator_id(), str)
    clone = pickle.loads(pickle.dumps(c))  # travels to the actors un-initialised (Q16)
    assert clone.get_world_size() == 2 and clone.get_self_rank() is None and clone._comm is None
    with c.send_stream, c.recv_stream:
        pass


@pytest.mark.parametrize("use_streams", [False, True])
def test_p2p_send_recv_sizes(actors, use_streams):
    """Ping-pong of fp16 tensors 1 KB .. 8 MB (config 3 shapes, incl. the 100 KB default of
    compiled_graph_gpu_microbenchmark.py:427)."""
    a = actors(2, use_communication_streams=use_streams)
    for nbytes in (1 << 10, 100_000, 1 << 20, (8 << 20) + 2):
        numel = nbytes // 2
        x = torch.randn(numel, generator=torch.Generator().manual_seed(nbytes)).to(torch.float16)

        def f(r, c):
            if r == 0:
                t = x.to(a.dev(0))
                c.send(t, 1)
                back = c.recv((numel,), torch.float16, 1, _alloc(a.dev(0)))
                c._recv_stream.synchronize()
                return back.cpu()
            got = c.recv((numel,), torch.float16, 0, _alloc(a.dev(1)))
            c._recv_stream.synchronize()
            c.send(got, 0)
            c._send_stream.synchronize()
            return got.cpu()

        out = a.run(f)
        assert torch.equal(out[0], x) and torch.equal(out[1], x)


@pytest.mark.parametrize("world", [2, 3])
def test_collectives_all_ops_torch_equal_fp16(actors, world):
    """test_torch_tensor_dag.py:1348-1459: every collective x every reduce op; bit exact at
    world 2 (single add), fp32-accumulated oracle at world 3."""
    from enum import Enum

    class CgraphReduceOp(Enum):  # same numbering as ray.experimental.util.types.ReduceOp
        SUM = 0
        PRODUCT = 1
        MAX = 2
        MIN = 3
        AVG = 4

    a = actors(world)
    shape = (4 * world, 6)
    xs = [(1.0 + 0.1 * torch.randn(shape, generator=torch.Generator().manual_seed(r))).to(torch.float16)
          for r in range(world)]
    np_in = [x.numpy() for x in xs]
    for op in CgraphReduceOp:
        def f(r, c):
            s = xs[r].to(a.dev(r))
            out = torch.empty_like(s)
            c.allreduce(s, out, op)
            rs = torch.empty((shape[0] // world, shape[1]), dtype=s.dtype, device=s.device)
            c.reducescatter(s, rs, op)
            return out.cpu().numpy(), rs.cpu().numpy()

        res = a.run(f)
        want = O.reduce_rank_ascending(np_in, O.CGRAPH_TO_COLLECTIVE_OP[op.value], accumulate="fp32")
        step = shape[0] // world
        for r in range(world):
            assert np.array_equal(res[r][0], want), op
            assert np.array_equal(res[r][1], want[r * step:(r + 1) * step]), op
        if world == 2 and op != CgraphReduceOp.AVG:
            native = O.cgraph_allreduce(np_in, op.value)[0]  # reference arithmetic in fp16
            assert np.array_equal(res[0][0], native), op

    def g(r, c):
        s = xs[r].to(a.dev(r))
        out = torch.empty((shape[0] * world, shape[1]), dtype=s.dtype, device=s.device)
        c.allgather(s, out)
        return out.cpu().numpy()

    cat = O.cgraph_allgather(np_in)[0]
    for got in a.run(g):
        assert np.array_equal(got, cat)
    # dtype mismatch assertion (nccl_group.py:253-257)
    with pytest.raises(AssertionError):
        a.comms[0].allreduce(torch.ones(2, device=a.dev(0)), torch.ones(2, device=a.dev(0), dtype=torch.float16), 0)
    with pytest.raises(ValueError):
        a.comms[0].allreduce(torch.ones(2, device=a.dev(0)), torch.ones(2, device=a.dev(0)), "nonsense")


def test_tensor_channel_dynamic_static_direct(actors):
    from ray_b200.channel import TorchTensorAcceleratorChannel

    a = actors(2)
    # dynamic shapes, list of tensors with mixed dtypes
    chans = [TorchTensorAcceleratorChannel(a.comms[r], 0, [1]) for r in range(2)]
    payloads = [[torch.randn(3, 5), torch.arange(7, dtype=torch.int64)], [torch.randn(11).to(torch.bfloat16)]]
    for msg in payloads:
        def f(r, c):
            if r == 0:
                chans[0].write([t.to(a.dev(0)) for t in msg])
                return None
            return [t.cpu() for t in chans[1].read()]

        got = a.run(f)[1]
        assert len(got) == len(msg) and all(torch.equal(g, m) for g, m in zip(got, msg))
    # static shape + direct return: metadata once, later mismatch is a writer-side ValueError (Q14)
    st = [TorchTensorAcceleratorChannel(a.comms[r], 0, [1], static_shape=True, direct_return=True) for r in range(2)]
    for i in range(3):
        x = torch.full((1000,), float(i), dtype=torch.float16)

        def f(r, c):
            if r == 0:
                st[0].write(x.to(a.dev(0)))
                return None
            return st[1].read().cpu()

        assert torch.equal(a.run(f)[1], x)
    with pytest.raises(ValueError, match="Expected torch.Tensors with shapes"):
        st[0].write(torch.zeros(5, device=a.dev(0), dtype=torch.float16))
    with pytest.raises(ValueError, match="_direct_return"):
        st[0].write([1, 2, 3])


@pytest.mark.parametrize("host_sync", [False, True])
def test_destroy_from_another_thread_unblocks_recv_and_raises(actors, host_sync):
    """compiled_dag_node.py:2157-2199 teardown: destroy() while the reader waits for data.  With
    host_sync=True the reader sits inside recv() like the reference's _NcclGroup; in the default
    event mode recv() returns at once and the reader sits in wait() on the tensor's event."""
    from ray_b200.channel import RayChannelError

    a = actors(2, host_sync=host_sync)
    reader = a.comms[1]
    result = {}

    def blocked():
        with torch.cuda.device(a.devices[1]), torch.cuda.stream(torch.cuda.Stream(a.devices[1])):
            reader._recv_stream = torch.cuda.current_stream()
            try:
                t0 = time.time()
                t = reader.recv((16,), torch.float32, 0, _alloc(a.dev(1)))
                result["recv_s"] = time.time() - t0
                reader.wait(t)
                result["err"] = None
            except RayChannelError as e:
                result["err"] = e

    t = threading.Thread(target=blocked)
    t.start()
    time.sleep(0.5)
    t0 = time.time()
    reader.destroy()  # from the "monitor" thread
    t.join(10)
    assert not t.is_alive() and time.time() - t0 < 8
    assert isinstance(result.get("err"), RayChannelError)
    if not host_sync:
        assert result["recv_s"] < 0.2, "recv() must not block the host in event mode"
    reader.destroy()  # idempotent
    with pytest.raises(RayChannelError):
        reader.send(torch.ones(1, device=a.dev(1)), 0)
    with pytest.raises(RayChannelError):
        reader.allreduce(torch.ones(1, device=a.dev(1)), torch.ones(1, device=a.dev(1)), 0)


def test_overlap_recv_does_not_block_the_host_and_is_event_guarded(actors):
    """overlap_gpu_communication (test_torch_tensor_dag.py overlap cases, dag_operation_future.py:
    101-133): recv is enqueued on the receive stream and returns immediately -- the host goes on
    to launch compute -- and the returned tensor carries the event a consumer stream waits on."""
    a = actors(2, use_communication_streams=True)
    numel = 1 << 20
    x = torch.randn(numel, generator=torch.Generator().manual_seed(5))

    def f(r, c):
        if r == 0:
            time.sleep(0.4)  # the receiver posts its recv long before the data exists
            c.send(x.to(a.dev(0)), 1)
            c._send_stream.synchronize()
            return None
        t0 = time.time()
        got = c.recv((numel,), torch.float32, 0, _alloc(a.dev(1)))
        dt = time.time() - t0
        busy = torch.ones(1 << 20, device=a.dev(1))
        for _ in range(10):  # host keeps launching compute while the recv kernel waits for its peer
            busy = busy * 1.0001
        launched_after = time.time() - t0
        assert got._b200_ready is not None
        y = got * 2  # current stream already waits on the event: safe without a host sync
        torch.cuda.current_stream().synchronize()
        return dt, launched_after, y.cpu()

    dt, launched_after, y = a.run(f)[1]
    assert dt < 0.2 and launched_after < 0.3, (dt, launched_after)
    assert torch.equal(y, x * 2)


def test_multi_reader_channel_uses_one_broadcast(actors):
    """A channel that spans the whole group and has several readers moves its payload with ONE
    broadcast collective instead of a send per reader (the reference's TODO at
    torch_tensor_accelerator_channel.py:587-590)."""
    from ray_b200.channel import TorchTensorAcceleratorChannel

    world = 3
    a = actors(world)
    chans = [TorchTensorAcceleratorChannel(a.comms[r], 0, [1, 2]) for r in range(world)]
    assert all(ch._use_broadcast for ch in chans)
    msg = [torch.randn(1000, 7), torch.arange(33, dtype=torch.int32)]

    def f(r, c):
        if r == 0:
            before = c.comm.launch_count
            chans[0].write([t.to(a.dev(0)) for t in msg])
            return c.comm.launch_count - before
        return [t.cpu() for t in chans[r].read()]

    out = a.run(f)
    assert out[0] == 2 + 2, "2 header sends + ONE broadcast per tensor"
    for r in (1, 2):
        assert all(torch.equal(g, m) for g, m in zip(out[r], msg))


@pytest.mark.parametrize("world", [2, 3])
def test_collective_operation_execute_matches_oracle(actors, world):
    """_CollectiveOperation.execute (dag/collective_node.py:176-248) through the B200
    communicator: output allocation, dim-0 layouts, multi-tensor all-reduce in one launch."""
    from ray_b200.channel import AllGatherOp, AllReduceOp, ReduceScatterOp, execute_collective

    a = actors(world)
    d0 = 2 * world
    xs = [torch.randn(d0, 4, generator=torch.Generator().manual_seed(r)) for r in range(world)]
    ys = [torch.randn(33, generator=torch.Generator().manual_seed(50 + r)) for r in range(world)]

    def f(r, c):
        x, y = xs[r].to(a.dev(r)), ys[r].to(a.dev(r))
        before = c.comm.launch_count
        multi = execute_collective(c, AllReduceOp(), x, y)
        launches = c.comm.launch_count - before
        return (execute_collective(c, AllGatherOp(), x).cpu().numpy(),
                execute_collective(c, AllReduceOp(), x).cpu().numpy(),
                execute_collective(c, ReduceScatterOp(), x).cpu().numpy(),
                [m.cpu().numpy() for m in multi], launches, x.cpu().numpy())

    res = a.run(f)
    np_x, np_y = [x.numpy() for x in xs], [y.numpy() for y in ys]
    for r in range(world):
        ag, ar, rs, multi, launches, x_after = res[r]
        assert np.array_equal(ag, O.cgraph_allgather(np_x)[r])
        assert np.array_equal(ar, O.cgraph_allreduce(np_x, 0)[r])
        assert np.array_equal(rs, O.cgraph_reducescatter(np_x, 0)[r])
        assert np.array_equal(multi[0], O.cgraph_allreduce(np_x, 0)[r])
        assert np.array_equal(multi[1], O.cgraph_allreduce(np_y, 0)[r])
        assert launches == 1, "the tensor list must be reduced by a single kernel launch"
        assert np.array_equal(x_after, np_x[r]), "inputs of an out-of-place collective are untouched"
