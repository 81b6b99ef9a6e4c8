"""Round-2 tuning sweeps (one process, one rank per GPU, CUDA-graph replay, device-timed).

    python scripts/r02_tune.py --world 2 --what allreduce,sendrecv,allgather [--quick]

allreduce : phase-by-phase kernels vs the chunk-pipelined ones (allreduce_pipe.cu) over
            chunk size / copy CTAs / reduce CTAs, on ordinary tensors
sendrecv  : ld/st p2p kernel vs the TMA bulk-copy kernel
allgather : staged all-gather vs the pull kernel over copy / pull CTAs
Output: one line per measurement; the chosen defaults are recorded in profiles/r02/.
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch

from ray_b200 import _native as N
from ray_b200.testing import LocalGroup
from scripts.bw_sweep import time_graphs

MiB = 1 << 20


def set_all(g, param, value):
    for c in g.comms:
        c.set_param(param, value)


def allreduce(g, args):
    n = g.world_size
    factor = 2 * (n - 1) / n
    sizes = [16 * MiB, 64 * MiB, 256 * MiB] if args.quick else [16 * MiB, 32 * MiB, 64 * MiB, 128 * MiB, 256 * MiB, 1024 * MiB]
    for dtype in (torch.float32,):
        for size in sizes:
            numel = size // 4
            xs = [torch.ones(numel, dtype=dtype, device=g.device(r)) for r in range(n)]
            iters = 20 if size <= 64 * MiB else 6

            def run(label, algo):
                us = time_graphs(g, lambda c, r: c.allreduce(xs[r], N.SUM, algo=algo), iters)
                print(f"allreduce n={n} {size >> 20:5d} MiB {label:44s} {us:9.1f} us  busbw={size / us / 1e3 * factor:7.1f} GB/s",
                      flush=True)

            set_all(g, N.PARAM_PIPE_MIN_BYTES, 1 << 40)  # AUTO without the pipeline = round-1 behaviour
            run("staged auto (r01 path)", N.ALGO_AUTO)
            set_all(g, N.PARAM_PIPE_MIN_BYTES, -1)
            variants = [("pull", 3)] if n == 2 else []
            if g.has_multicast and n > 2:
                variants.append(("nvls", 1))
            if args.peer:
                variants.append(("peer", 2))
            for vname, v in variants:
                set_all(g, N.PARAM_PIPE_VARIANT, v)
                if vname == "pull":
                    grid = [(1, 16, 16), (1, 16, 24), (1, 16, 32), (1, 16, 48), (1, 16, 64), (1, 32, 32), (1, 32, 48), (2, 16, 32)]
                else:
                    grid = [(1, 16, 64), (2, 16, 64), (4, 16, 64), (4, 16, 32), (4, 8, 64), (4, 16, 96), (8, 16, 64), (8, 16, 32)]
                if args.quick:
                    grid = grid[1:4]
                for chunk_mib, copy, red in grid:
                    set_all(g, N.PARAM_PIPE_CHUNK_BYTES, chunk_mib * MiB)
                    set_all(g, N.PARAM_PIPE_COPY_CTAS, copy)
                    set_all(g, N.PARAM_PIPE_RED_CTAS, red)
                    run(f"pipe {vname} chunk={chunk_mib}MiB copy={copy} red={red}", N.ALGO_PIPE)
            for p in (N.PARAM_PIPE_VARIANT, N.PARAM_PIPE_CHUNK_BYTES, N.PARAM_PIPE_COPY_CTAS, N.PARAM_PIPE_RED_CTAS):
                set_all(g, p, -1)
            run("AUTO (defaults)", N.ALGO_AUTO)
            del xs


def sendrecv(g, args):
    n = g.world_size
    sizes = [MiB, 4 * MiB, 32 * MiB, 256 * MiB] if args.quick else [256 << 10, MiB, 4 * MiB, 16 * MiB, 32 * MiB, 64 * MiB, 256 * MiB, 1024 * MiB]
    for size in sizes:
        xs = [torch.ones(size // 4, device=g.device(r)) for r in range(n)]
        iters = 20 if size <= 64 * MiB else 6
        call = lambda c, r: (c.send(xs[0], 1) if r == 0 else (c.recv(xs[1], 0) if r == 1 else None))  # noqa: E731
        for label, v in (("ld/st", 0), ("bulk", -1)):
            set_all(g, N.PARAM_P2P_BULK_MIN_CHUNK, v)
            us = time_graphs(g, call, iters)
            print(f"sendrecv n={n} {size / MiB:8.2f} MiB {label:16s} {us:9.1f} us  {size / us / 1e3:7.1f} GB/s", flush=True)
        del xs
    set_all(g, N.PARAM_P2P_BULK_MIN_CHUNK, -1)


def allgather(g, args):
    n = g.world_size
    for total in ([16 * MiB, 64 * MiB, 256 * MiB, 1024 * MiB]):
        per = total // n // 4
        xs = [torch.ones(per, device=g.device(r)) for r in range(n)]
        outs = [torch.empty(per * n, device=g.device(r)) for r in range(n)]
        iters = 20 if total <= 64 * MiB else 6
        call = lambda c, r: c.allgather_into(outs[r], xs[r])  # noqa: E731
        configs = [("staged (r01)", 0, -1, -1)] + [(f"pull copy={cp} pull={pl}", -1, cp, pl) for cp, pl in
                                                   ((8, 16), (16, 16), (16, 32), (16, 48), (32, 32), (8, 32))]
        for label, mn, cp, pl in configs:
            set_all(g, N.PARAM_AG_PULL_MIN_BYTES, mn)
            set_all(g, N.PARAM_PIPE_COPY_CTAS, cp)
            set_all(g, N.PARAM_PIPE_RED_CTAS, pl)
            us = time_graphs(g, call, iters)
            print(f"allgather n={n} total {total >> 20:5d} MiB {label:24s} {us:9.1f} us  busbw={per * 4 * n / us / 1e3 * (n - 1) / n:7.1f} GB/s",
                  flush=True)
        del xs, outs
    for p in (N.PARAM_AG_PULL_MIN_BYTES, N.PARAM_PIPE_COPY_CTAS, N.PARAM_PIPE_RED_CTAS):
        set_all(g, p, -1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--world", type=int, default=2)
    ap.add_argument("--what", default="allreduce,sendrecv")
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--peer", action="store_true", help="also sweep the peer ld/st pipeline")
    args = ap.parse_args()
    g = LocalGroup(args.world, timeout_ms=20000, staging_bytes=256 << 20, inbox_bytes=32 << 20)
    print(f"# world={args.world} devices={g.devices} shared={g.shared_gpu} multicast={g.has_multicast}", flush=True)
    for what in args.what.split(","):
        {"allreduce": allreduce, "sendrecv": sendrecv, "allgather": allgather}[what](g, args)
    g.destroy()


if __name__ == "__main__":
    main()
