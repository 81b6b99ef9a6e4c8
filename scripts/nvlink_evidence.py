"""Per-kernel evidence for the NVLink kernels (one process, one rank per GPU).

For every collective kernel of the library: device time per launch (CUDA events around a loop of
launches, max over ranks), the nccl-tests bus bandwidth, and the NVLink bytes that actually crossed
the links of GPU 0 during the loop, read from the driver's NVLink counters through NVML
(NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX / _RX, KiB, all links; RAW = including protocol overhead).
This is the multi-GPU counterpart of an ncu capture: ncu serialises kernels, and the kernels of a
collective wait for each other across GPUs, so they cannot be replayed one at a time.

    python scripts/nvlink_evidence.py --world 2 [--ncu-range CASE]   # CASE: run one case inside
                                                                      # cudaProfilerStart/Stop for
                                                                      # ncu --replay-mode app-range
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pynvml
import torch

from ray_b200 import _native as N
from ray_b200.testing import LocalGroup

MiB = 1 << 20
ap = argparse.ArgumentParser()
ap.add_argument("--world", type=int, default=2)
ap.add_argument("--ncu-range", default=None)
ap.add_argument("--out", default=None)
args = ap.parse_args()
n = args.world
g = LocalGroup(n, timeout_ms=20000, staging_bytes=256 << 20, inbox_bytes=32 << 20, heap_bytes=80 << 20)
pynvml.nvmlInit()
h0 = pynvml.nvmlDeviceGetHandleByIndex(g.devices[0])


ALL_LINKS = 0xFFFFFFFF  # scopeId: UINT_MAX = sum over the GPU's 18 links


def nvlink_kib():
    ids = [pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX,
           pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_RAW_TX, pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_RAW_RX]
    try:
        vals = pynvml.nvmlDeviceGetFieldValues(h0, [(i, ALL_LINKS) for i in ids])
        if any(v.nvmlReturn != 0 for v in vals):
            raise RuntimeError("scope not supported")
        return [int(v.value.ullVal) for v in vals]
    except Exception:
        tot = [0, 0, 0, 0]
        for link in range(18):
            vals = pynvml.nvmlDeviceGetFieldValues(h0, [(i, link) for i in ids])
            for k, v in enumerate(vals):
                if v.nvmlReturn == 0:
                    tot[k] += int(v.value.ullVal)
        return tot


def cases():
    def ar(size, algo, variant=-1, dtype=torch.float32):
        xs = [torch.ones(size // torch.empty((), dtype=dtype).element_size(), dtype=dtype, device=g.device(r)) for r in range(n)]

        def call(c, r):
            c.allreduce(xs[r], N.SUM, algo=algo)
        return call, size, 2 * (n - 1) / n, dict(variant=variant)

    yield "allreduce_ll_kernel 4KiB", ar(4096, N.ALGO_LL)
    yield "allreduce_oneshot_kernel 256KiB", ar(256 << 10, N.ALGO_ONESHOT)
    yield "allreduce_twoshot_kernel 16MiB", ar(16 * MiB, N.ALGO_TWOSHOT)
    if g.has_multicast:
        yield "allreduce_twoshot_kernel<NVLS> 64MiB", ar(64 * MiB, N.ALGO_NVLS)
    if n == 2:
        yield "allreduce_pull_kernel 64MiB", ar(64 * MiB, N.ALGO_PIPE, 3)
        yield "allreduce_pull_kernel 256MiB", ar(256 * MiB, N.ALGO_PIPE, 3)
    else:
        if g.has_multicast:
            yield "allreduce_pipe_kernel<NVLS> 256MiB", ar(256 * MiB, N.ALGO_PIPE, 1)
        yield "allreduce_pipe_kernel<peer> 64MiB", ar(64 * MiB, N.ALGO_PIPE, 2)
    per = 64 * MiB // n // 4
    xs = [torch.ones(per, device=g.device(r)) for r in range(n)]
    ys = [torch.empty(per * n, device=g.device(r)) for r in range(n)]
    yield "allgather_pull_kernel 64MiB total", ((lambda c, r: c.allgather_into(ys[r], xs[r])), per * 4 * n, (n - 1) / n, {})
    small = [torch.ones(64 << 10, device=g.device(r)) for r in range(n)]
    smo = [torch.empty((64 << 10) * n, device=g.device(r)) for r in range(n)]
    yield "allgather_kernel 256KiB/rank", ((lambda c, r: c.allgather_into(smo[r], small[r])), (256 << 10) * n, (n - 1) / n, {})
    ins = [torch.ones(per * n, device=g.device(r)) for r in range(n)]
    outs = [torch.empty(per, device=g.device(r)) for r in range(n)]
    yield "reducescatter_kernel 64MiB total", ((lambda c, r: c.reducescatter_from(outs[r], ins[r], N.SUM)), per * 4 * n, (n - 1) / n, {})
    b = [torch.ones(64 * MiB // 4, device=g.device(r)) for r in range(n)]
    yield "broadcast_kernel 64MiB", ((lambda c, r: c.broadcast(b[r], 0)), 64 * MiB, 1.0, {})
    red = [torch.ones(16 * MiB // 4, device=g.device(r)) for r in range(n)]
    yield "reduce_kernel 16MiB", ((lambda c, r: c.reduce(red[r], 0, N.SUM)), 16 * MiB, 1.0, {})
    p2p = [torch.ones(64 * MiB // 4, device=g.device(r)) for r in range(n)]
    yield "p2p_bulk_kernel send+recv 64MiB", ((lambda c, r: c.send(p2p[0], 1) if r == 0 else (c.recv(p2p[1], 0) if r == 1 else None)), 64 * MiB, 1.0, {})
    sm = [torch.ones(4096 // 4, device=g.device(r)) for r in range(n)]
    yield "p2p_kernel send+recv 4KiB", ((lambda c, r: c.send(sm[0], 1) if r == 0 else (c.recv(sm[1], 0) if r == 1 else None)), 4096, 1.0, {})
    gr = [torch.ones(25 * MiB // 4, device=g.device(r)) for r in range(n)]
    yield "grad_allreduce_kernel 25MiB fp32 bucket, bf16 wire", ((lambda c, r: c.grad_allreduce(gr[r], 1.0 / n, torch.bfloat16)), 25 * MiB // 2, 2 * (n - 1) / n, {})
    dst = torch.empty(64 * MiB, dtype=torch.uint8, device=g.device(1 % n))
    yield "get_bulk_kernel (one-sided) 64MiB", ((lambda c, r: c.get(dst, 0, 0) if r == 1 % n else None), 64 * MiB, 1.0, {})
    yield "barrier_kernel", ((lambda c, r: c.barrier()), 0, 0.0, {})


rows = []
for name, (call, size, factor, opt) in cases():
    if args.ncu_range and args.ncu_range not in name:
        continue
    for c in g.comms:
        c.set_param(N.PARAM_PIPE_VARIANT, opt.get("variant", -1))
    iters = 200 if size <= MiB else (30 if size <= 64 * MiB else 10)
    for _ in range(3):
        g.run(call)
    if args.ncu_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        g.run(call)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print("ncu range done:", name)
        continue
    torch.cuda.synchronize()
    k0 = nvlink_kib()
    starts, ends = [], []
    for r in range(n):
        with torch.cuda.device(g.devices[r]), torch.cuda.stream(g.streams[r]):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            starts.append(s)
            ends.append(e)
    for _ in range(iters):
        for r, c in enumerate(g.comms):
            with torch.cuda.device(g.devices[r]), torch.cuda.stream(g.streams[r]):
                call(c, r)
    for r in range(n):
        with torch.cuda.device(g.devices[r]), torch.cuda.stream(g.streams[r]):
            ends[r].record()
    g.synchronize()
    time.sleep(0.05)
    k1 = nvlink_kib()
    us = max(s.elapsed_time(e) for s, e in zip(starts, ends)) * 1e3 / iters
    tx, rx, rtx, rrx = [(b - a) * 1024 / iters if a >= 0 and b >= 0 else None for a, b in zip(k0, k1)]
    row = {"kernel": name, "world": n, "bytes": size, "us_per_launch": round(us, 2),
           "busbw_gbs": round(size / us / 1e3 * factor, 1) if size else None,
           "nvlink_tx_bytes_per_launch": tx, "nvlink_rx_bytes_per_launch": rx,
           "nvlink_tx_gbs": round(tx / us / 1e3, 1) if tx else None, "nvlink_rx_gbs": round(rx / us / 1e3, 1) if rx else None,
           "nvlink_raw_tx_gbs": round(rtx / us / 1e3, 1) if rtx else None, "nvlink_raw_rx_gbs": round(rrx / us / 1e3, 1) if rrx else None,
           "frac_of_900": round(max(tx or 0, rx or 0) / us / 1e3 / 900, 3) if (tx or rx) else None}
    rows.append(row)
    print(json.dumps(row), flush=True)
for c in g.comms:
    c.set_param(N.PARAM_PIPE_VARIANT, -1)
if args.out and rows:
    json.dump(rows, open(args.out, "w"), indent=1)
g.destroy()
