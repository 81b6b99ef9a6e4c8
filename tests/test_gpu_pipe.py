"""GPU parity tests of the chunk-pipelined all-reduce kernels (allreduce_pipe.cu: TMA bulk-copy
roles + reduce role synchronised by per-chunk flags) against the rank-ascending oracle.

Peer ld/st and pull variants are bit exact against the oracle for every dtype; the NVLS variant
(multi-GPU boxes only) is exact on integer-valued data and within 1e-6 * sum|x| otherwise.
"""
import numpy as np
import pytest
import torch

from oracle import collective_oracle as O

pytestmark = pytest.mark.gpu

MiB = 1 << 20
# bytes per rank: one unit, sub-tile, tile boundary +-, one chunk exactly, chunk +- one unit,
# several chunks with a ragged tail
SIZES = [16, 16 * 1023, 16 << 10, (16 << 10) + 16, MiB - 16, MiB, MiB + 16, 3 * MiB + 16 * 77, 5 * MiB]


@pytest.fixture(scope="module")
def pipe_groups(native_lib):
    from ray_b200.testing import LocalGroup

    cache = {}

    def get(n):
        if n not in cache:
            cache[n] = LocalGroup(n, timeout_ms=20000, staging_bytes=40 << 20, inbox_bytes=2 << 20)
        return cache[n]

    yield get
    for g in cache.values():
        g.destroy()


def _variants(g, world):
    from ray_b200 import _native as N

    out = [("peer", 2)]
    if world == 2:
        out.append(("pull", 3))
    if g.has_multicast:
        out.append(("nvls", 1))
    return out, N


def _rand(numel, dtype, seed):
    gen = torch.Generator().manual_seed(seed)
    if dtype.is_floating_point:
        return torch.randn(numel, generator=gen).to(dtype)
    return torch.randint(-1000, 1000, (numel,), generator=gen).to(dtype)


def _np(t):
    if t.dtype == torch.bfloat16:
        import ml_dtypes

        return t.cpu().view(torch.uint16).numpy().view(ml_dtypes.bfloat16)
    return t.cpu().numpy()


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_pipelined_allreduce_matches_oracle(pipe_groups, world):
    g = pipe_groups(world)
    variants, N = _variants(g, world)
    cases = [(torch.float32, N.SUM), (torch.int32, N.SUM), (torch.bfloat16, N.SUM), (torch.float64, N.MAX),
             (torch.uint8, N.SUM), (torch.float32, N.AVG)]
    for vname, vcode in variants:
        for c in g.comms:
            c.set_param(N.PARAM_PIPE_VARIANT, vcode)
        try:
            for dtype, op in cases:
                if vname == "nvls" and not (dtype in (torch.float32, torch.bfloat16) and op in (N.SUM, N.AVG)):
                    continue
                es = torch.empty((), dtype=dtype).element_size()
                for nbytes in SIZES:
                    numel = nbytes // es
                    host = [_rand(numel, dtype, 1000 * world + 17 * r + nbytes % 97) for r in range(world)]
                    if vname == "nvls":  # integer-valued: any summation order is exact
                        host = [(h.float() * 4).round().clamp(-64, 64).to(dtype) for h in host]
                    xs = [h.to(g.device(r)) for r, h in enumerate(host)]
                    g.run(lambda c, r: c.allreduce(xs[r], op, algo=N.ALGO_PIPE))
                    half = dtype in (torch.bfloat16, torch.float16)
                    want = O.reduce_rank_ascending([_np(h) for h in host], op,
                                                   accumulate="fp32" if half else "native")
                    for r in range(world):
                        got = _np(xs[r])
                        if vname == "nvls":
                            # the switch may return +0.0 where IEEE gives -0.0 (observed): compare values
                            assert np.array_equal(got.astype(np.float64), np.asarray(want).astype(np.float64)), \
                                (vname, world, dtype, op, nbytes, r)
                            assert np.array_equal(got.view(np.uint8), _np(xs[0]).view(np.uint8))  # replicas agree
                        else:
                            assert np.array_equal(got.view(np.uint8), np.asarray(want).view(np.uint8)), \
                                (vname, world, dtype, op, nbytes, r)
        finally:
            for c in g.comms:
                c.set_param(N.PARAM_PIPE_VARIANT, -1)


@pytest.mark.parametrize("world", [2, 4])
def test_pipelined_allreduce_out_of_place_and_back_to_back(pipe_groups, world):
    """Out-of-place operands (the Compiled-Graph allreduce is out of place, nccl_group.py:293-312)
    and a sequence of launches that alternates slots and mixes kernels: the slot-rotation argument
    must hold across pipelined and phase-by-phase launches."""
    from ray_b200 import _native as N

    g = pipe_groups(world)
    numel = (2 * MiB + 4096) // 4
    host = [_rand(numel, torch.float32, 31 * r + world) for r in range(world)]
    want = O.reduce_rank_ascending([h.numpy() for h in host], N.SUM)
    ins = [h.to(g.device(r)) for r, h in enumerate(host)]
    outs = [torch.zeros_like(x) for x in ins]
    small = [torch.full((1000,), float(r + 1), device=g.device(r)) for r in range(world)]
    for rep in range(6):
        for o in outs:
            o.zero_()
        g.run(lambda c, r: c.allreduce(ins[r], N.SUM, out=outs[r], algo=N.ALGO_PIPE))
        for r in range(world):
            got = outs[r].cpu().numpy()
            if g.has_multicast and world > 2:  # NVLS roles: the switch picks the summation order
                bound = 1e-6 * np.sum([np.abs(h.numpy().astype(np.float64)) for h in host], axis=0)
                assert np.all(np.abs(got.astype(np.float64) - want.astype(np.float64)) <= bound), (world, rep)
                assert np.array_equal(got, outs[0].cpu().numpy())  # replicas bit-identical
            else:
                assert np.array_equal(got, want), (world, rep)
            assert torch.equal(ins[r].cpu(), host[r])  # inputs untouched
        if rep % 2:
            ys = [s.clone() for s in small]
            g.run(lambda c, r: c.allreduce(ys[r], N.SUM))
            assert all(torch.all(y == sum(range(1, world + 1))) for y in ys)


def test_auto_picks_the_pipeline_for_large_aligned_messages(pipe_groups):
    """AUTO: ordinary 16-byte aligned tensors from 16 MiB on go through the pipelined kernels
    (pull at world 2); a misaligned view of the same size falls back to the staged kernels and
    still produces the same bits."""
    from ray_b200 import _native as N

    g = pipe_groups(2)
    numel = (20 * MiB) // 4
    host = [_rand(numel + 1, torch.float32, 5 + r) for r in range(2)]
    want = O.reduce_rank_ascending([h[:numel].numpy() for h in host], N.SUM)
    xs = [h.to(g.device(r)) for r, h in enumerate(host)]
    g.run(lambda c, r: c.allreduce(xs[r][:numel], N.SUM))
    for r in range(2):
        assert np.array_equal(xs[r][:numel].cpu().numpy(), want)
        assert xs[r][numel].item() == host[r][numel].item()  # the element past the end is untouched
    ys = [h.to(g.device(r)) for r, h in enumerate(host)]
    want_mis = O.reduce_rank_ascending([h[1:].numpy() for h in host], N.SUM)
    g.run(lambda c, r: c.allreduce(ys[r][1:], N.SUM))  # 4-byte offset: not 16-byte aligned
    for r in range(2):
        assert np.array_equal(ys[r][1:].cpu().numpy(), want_mis)
    with pytest.raises(N.B200Error):
        g.comms[0].allreduce(ys[0][1:], N.SUM, algo=N.ALGO_PIPE)


@pytest.mark.parametrize("world", [2, 8])
def test_pipeline_tuning_parameters_do_not_change_results(pipe_groups, world):
    from ray_b200 import _native as N

    g = pipe_groups(world)
    numel = (4 * MiB + 16 * 5) // 4
    host = [_rand(numel, torch.float32, 77 + r) for r in range(world)]
    want = O.reduce_rank_ascending([h.numpy() for h in host], N.SUM)
    try:
        for chunk, copy_ctas, red_ctas in ((1 * MiB, 1, 2), (2 * MiB, 2, 3), (1 * MiB, 4, 1), (3 * MiB, 2, 5)):
            for c in g.comms:
                c.set_param(N.PARAM_PIPE_CHUNK_BYTES, chunk)
                c.set_param(N.PARAM_PIPE_COPY_CTAS, copy_ctas)
                c.set_param(N.PARAM_PIPE_RED_CTAS, red_ctas)
            xs = [h.to(g.device(r)) for r, h in enumerate(host)]
            g.run(lambda c, r: c.allreduce(xs[r], N.SUM, algo=N.ALGO_PIPE))
            for r in range(world):
                got = xs[r].cpu().numpy()
                if g.has_multicast and world > 2:  # NVLS roles: the switch picks the summation order
                    bound = 1e-6 * np.sum([np.abs(h.numpy().astype(np.float64)) for h in host], axis=0)
                    assert np.all(np.abs(got.astype(np.float64) - want.astype(np.float64)) <= bound)
                    assert np.array_equal(got, xs[0].cpu().numpy())
                else:
                    assert np.array_equal(got, want), (world, chunk, copy_ctas, red_ctas)
    finally:
        for c in g.comms:
            for p in (N.PARAM_PIPE_CHUNK_BYTES, N.PARAM_PIPE_COPY_CTAS, N.PARAM_PIPE_RED_CTAS):
                c.set_param(p, -1)


@pytest.mark.parametrize("world", [2, 4])
def test_bulk_copy_send_recv_is_byte_exact(native_lib, world):
    """send/recv through the TMA bulk-copy kernel (p2p_bulk_kernel): sizes around the chunk and
    ring boundaries, a message several times the ring (flow control by ack flags), an eager send
    that completes before the receive is posted, and the mixed case where only one side's tensor
    is 16-byte aligned (that side uses the bulk kernel, the other the ld/st kernel -- one
    protocol)."""
    from ray_b200 import _native as N
    from ray_b200.testing import LocalGroup

    with LocalGroup(world, timeout_ms=20000, staging_bytes=2 << 20, inbox_bytes=8 << 20) as g:
        src, dst = 0, world - 1
        for nbytes in (512 << 10, (512 << 10) + 16, MiB + 4096, 8 * MiB, 8 * MiB + 16, 27 * MiB + 48):
            a = torch.randint(0, 255, (nbytes,), dtype=torch.uint8, device=g.device(src))
            b = torch.zeros(nbytes, dtype=torch.uint8, device=g.device(dst))
            before = g.comms[src].launch_count
            g.run(lambda c, r: c.send(a, dst) if r == src else (c.recv(b, src) if r == dst else None))
            assert g.comms[src].launch_count == before + 1
            assert torch.equal(a.cpu(), b.cpu()), nbytes
        # eager: 4 MiB fits the 8 MiB ring, the send kernel finishes with no receiver running
        a = torch.randint(0, 255, (4 * MiB,), dtype=torch.uint8, device=g.device(src))
        b = torch.zeros_like(a, device=g.device(dst))
        torch.cuda.synchronize()
        with torch.cuda.device(g.devices[src]), torch.cuda.stream(g.streams[src]):
            g.comms[src].send(a, dst)
        g.streams[src].synchronize()
        with torch.cuda.device(g.devices[dst]), torch.cuda.stream(g.streams[dst]):
            g.comms[dst].recv(b, src)
        g.synchronize()
        assert torch.equal(a.cpu(), b.cpu())
        # mixed mechanisms: misaligned receiver, then misaligned sender
        nbytes = 3 * MiB
        a = torch.randint(0, 255, (nbytes + 16,), dtype=torch.uint8, device=g.device(src))
        b = torch.zeros(nbytes + 16, dtype=torch.uint8, device=g.device(dst))
        g.run(lambda c, r: c.send(a[:nbytes], dst) if r == src else (c.recv(b[3:nbytes + 3], src) if r == dst else None))
        assert torch.equal(a[:nbytes].cpu(), b[3:nbytes + 3].cpu()) and b[:3].sum().item() == 0
        b.zero_()
        g.run(lambda c, r: c.send(a[5:nbytes + 5], dst) if r == src else (c.recv(b[:nbytes], src) if r == dst else None))
        assert torch.equal(a[5:nbytes + 5].cpu(), b[:nbytes].cpu())
        # the ld/st kernel alone gives the same bytes
        for c in g.comms:
            c.set_param(N.PARAM_P2P_BULK_MIN_CHUNK, 0)
        b.zero_()
        g.run(lambda c, r: c.send(a[:nbytes], dst) if r == src else (c.recv(b[:nbytes], src) if r == dst else None))
        assert torch.equal(a[:nbytes].cpu(), b[:nbytes].cpu())
        # ping-pong in both directions, bulk on both legs
        for c in g.comms:
            c.set_param(N.PARAM_P2P_BULK_MIN_CHUNK, -1)
        x = torch.randn(MiB, device=g.device(src))
        y = torch.zeros(MiB, device=g.device(dst))
        z = torch.zeros(MiB, device=g.device(src))

        def pingpong(c, r):
            if r == src:
                c.send(x, dst)
                c.recv(z, dst)
            elif r == dst:
                c.recv(y, src)
                c.send(y, src)

        for _ in range(3):
            g.run(pingpong)
            assert torch.equal(z.cpu(), x.cpu())


@pytest.mark.parametrize("world", [2, 3, 8])
def test_pull_allgather_is_byte_exact(pipe_groups, world):
    """all-gather through the pull kernel (TMA copy-in + bulk loads of every peer's slot straight
    into the caller's output tensors): sizes around the tile / chunk boundaries, separately
    allocated outputs and the Compiled-Graph concatenated layout, and the misaligned fallback."""
    from ray_b200 import _native as N

    g = pipe_groups(world)
    for nbytes in (4 * MiB, 4 * MiB + 16, 5 * MiB - 16, 6 * MiB + 16 * 1001):
        host = [torch.randint(0, 255, (nbytes,), dtype=torch.uint8, generator=torch.Generator().manual_seed(nbytes % 1000 + r))
                for r in range(world)]
        xs = [h.to(g.device(r)) for r, h in enumerate(host)]
        outs = [[torch.zeros(nbytes, dtype=torch.uint8, device=g.device(r)) for _ in range(world)] for r in range(world)]
        before = g.comms[0].launch_count
        g.run(lambda c, r: c.allgather(outs[r], xs[r]))
        assert g.comms[0].launch_count == before + 1
        for r in range(world):
            for p in range(world):
                assert torch.equal(outs[r][p].cpu(), host[p]), (world, nbytes, r, p)
        cat = [torch.zeros(world * nbytes, dtype=torch.uint8, device=g.device(r)) for r in range(world)]
        g.run(lambda c, r: c.allgather_into(cat[r], xs[r]))
        want = torch.cat(host)
        for r in range(world):
            assert torch.equal(cat[r].cpu(), want), (world, nbytes, r)
    # misaligned input: staged kernel, same bytes
    nbytes = 5 * MiB
    host = [torch.randint(0, 255, (nbytes + 1,), dtype=torch.uint8, generator=torch.Generator().manual_seed(9 + r))
            for r in range(world)]
    xs = [h.to(g.device(r)) for r, h in enumerate(host)]
    outs = [[torch.zeros(nbytes, dtype=torch.uint8, device=g.device(r)) for _ in range(world)] for r in range(world)]
    g.run(lambda c, r: c.allgather(outs[r], xs[r][1:]))
    for r in range(world):
        for p in range(world):
            assert torch.equal(outs[r][p].cpu(), host[p][1:])


@pytest.mark.parametrize("world", [3, 4])
def test_chunk_ring_handles_messages_larger_than_the_staging_slot_in_one_launch(pipe_groups, world):
    """n >= 3 pipeline with the slot used as a ring of chunks: a message several times the slot
    size goes through ONE launch (copy-in of chunk k waits for the copy-out of chunk k - R).  A
    chunk size that leaves fewer than 4 chunks in the slot turns the ring off, and the message is
    split into launches of as many whole chunks as the slot holds; that must give the same bits."""
    from ray_b200 import _native as N

    staging = 40 * MiB
    g = pipe_groups(world)
    nbytes = 97 * MiB + 16 * 3
    numel = nbytes // 4
    host = [(torch.arange(numel, dtype=torch.float32) % 1021) * (r + 1) - 3 * r for r in range(world)]
    want = sum(host)
    try:
        for chunk in (1 * MiB, 4 * MiB, 16 * MiB):
            ring = staging // chunk >= 4
            split = staging // chunk * chunk  # bytes per launch without the ring
            for c in g.comms:
                c.set_param(N.PARAM_PIPE_CHUNK_BYTES, chunk)
            xs = [h.to(g.device(r)) for r, h in enumerate(host)]
            before = g.comms[0].launch_count
            g.run(lambda c, r: c.allreduce(xs[r], N.SUM, algo=N.ALGO_PIPE))
            launches = g.comms[0].launch_count - before
            assert launches == (1 if ring else -(-nbytes // split)), (chunk, launches)
            for r in range(world):
                assert torch.equal(xs[r].cpu(), want), (world, chunk, r)
            del xs
    finally:
        for c in g.comms:
            c.set_param(N.PARAM_PIPE_CHUNK_BYTES, -1)


def test_pipe_variant_parameter_rejects_unknown_values(pipe_groups):
    """B200_PARAM_PIPE_VARIANT takes -1 (automatic), 1 (NVLS), 2 (peer) or 3 (pull); anything else,
    such as 0 for the removed push kernel, is refused instead of silently selecting another kernel."""
    from ray_b200 import _native as N

    c = pipe_groups(2).comms[0]
    try:
        for bad in (0, 4, -2):
            with pytest.raises(N.B200Error):
                c.set_param(N.PARAM_PIPE_VARIANT, bad)
        for good in (1, 2, 3, -1):
            c.set_param(N.PARAM_PIPE_VARIANT, good)
    finally:
        c.set_param(N.PARAM_PIPE_VARIANT, -1)
