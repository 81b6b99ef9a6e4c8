#!/usr/bin/env python
"""bench.py -- TorchTrainer-shaped ResNet-50 DDP step (BASELINE.json configs[1]) on N B200s.

    python bench.py --gpus 1 --steps 50 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...   # the reference's CPU path (gloo DDP on host cores)
    python bench.py --impl nccl ...        # comparator: stock torch DDP over NCCL (not the product)
    python bench.py ... --dump-outputs DIR # also write what the last timed step computed (.npy)

One step = forward + backward + Adam update of torchvision ResNet-50 (random init, synthetic
224x224 batch, bf16 autocast, per-GPU batch 32 as in release/train_tests/benchmark/config.py:15),
with the gradient synchronisation -- the hot path of this repository -- running in
libb200_collective.so through the b200 c10d backend and the fused bf16 gradient hook.
Rank 0 prints ONE JSON line (see DESIGN.md "Measurement").
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def log(msg):
    """Progress goes to stderr; stdout carries exactly one JSON line."""
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


METRIC = "TorchTrainer ResNet-50 DDP samples/sec"
UNIT = "samples/s"
FLOPS_PER_SAMPLE = 24.6e9  # fwd+bwd, 224x224 (SURVEY 8d; 3 x 8.2 GFLOP)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="b200", choices=["b200", "reference", "nccl"])
    p.add_argument("--batch", type=int, default=32, help="per-GPU batch")
    p.add_argument("--grad-wire", default="bf16", choices=["bf16", "f32", "none"],
                   help="wire dtype of the fused gradient hook; none = plain reducer all-reduce")
    p.add_argument("--no-sweep", action="store_true", help="skip the all-reduce bandwidth sweep (N>1)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-nccl-comparator", action="store_true", help="skip the in-line NCCL comparator leg (N>1)")
    p.add_argument("--profile", action="store_true",
                   help="under ncu: skip the end-to-end and sweep legs (numbers printed in this mode are not bench values)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last one computed as DIR/<name>.npy (GPU arms)")
    p.add_argument("--cpu-worker", default=None, help=argparse.SUPPRESS)
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        p.error("--dump-outputs applies to the GPU arms")
    return args


def env_rank():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._loop, daemon=True)

    def _loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = []
        for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
            if any(r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ----------------------------------------------------------------------------- model
def build(device, seed=0):
    import torch
    import torchvision

    torch.manual_seed(seed)
    model = torchvision.models.resnet50(weights=None).to(device)
    return model


def train_step(model, opt, x, y, device_type):
    import torch

    with torch.autocast(device_type, dtype=torch.bfloat16):
        loss = torch.nn.functional.cross_entropy(model(x), y)
    loss.backward()
    opt.step()
    opt.zero_grad(set_to_none=False)
    return loss


DUMP_PARAMS = 1 << 22  # parameters sampled by --dump-outputs: 16 MiB of the model's ~100 MiB


def dump_outputs(out_dir, model, loss):
    """Writes what one training step hands back: its loss (loss.npy), the updated parameters
    (params.npy: the same seeded sample of DUMP_PARAMS positions of all parameters flattened in
    model order, every run) and the BatchNorm running statistics (buffers.npy: every
    floating-point buffer, flattened).  float32."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    with torch.no_grad():
        flat = torch.cat([p.detach().reshape(-1).float() for p in model.parameters()])
        pick = np.random.default_rng(0).choice(flat.numel(), min(DUMP_PARAMS, flat.numel()), replace=False)
        params = flat[torch.from_numpy(np.sort(pick)).to(flat.device)].cpu().numpy()
        buffers = torch.cat([b.detach().reshape(-1).float() for b in model.buffers() if b.is_floating_point()])
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().reshape(1).cpu().numpy())
    np.save(os.path.join(out_dir, "params.npy"), params)
    np.save(os.path.join(out_dir, "buffers.npy"), buffers.cpu().numpy())


# ----------------------------------------------------------------------------- GPU arms
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP

    rank, local_rank, world = env_rank()
    if world != args.gpus and world > 1:
        args.gpus = world
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if "MASTER_ADDR" not in os.environ:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(free_port())

    pg = None
    if args.impl == "b200":
        from ray_b200 import train as b200_train
        from ray_b200 import _native as N

        N.load()  # fail loudly if the CUDA library is missing
        b200_train.setup_torch_process_group(b200_train.DEFAULT_GPU_BACKEND, rank, world, "env://")
        pg = dist.distributed_c10d._get_default_group()
    else:
        dist.init_process_group("cpu:gloo,cuda:nccl", rank=rank, world_size=world, device_id=device)

    log(f"process group up (impl={args.impl}, world={world}); building ResNet-50")
    model = build(device)
    # DDP is applied at world_size 1 too so the gradient-sync path (bucketing + hook) is on the
    # timed path at every N; TorchTrainer itself skips the wrap for a single worker.
    model = DDP(model, device_ids=[device], output_device=device)
    wire = {"bf16": torch.bfloat16, "f32": torch.float32}.get(args.grad_wire)
    if args.impl == "b200" and wire is not None:
        model.register_comm_hook(None, b200_train.b200_grad_hook(wire))
    elif args.impl == "nccl" and args.grad_wire == "bf16":
        from torch.distributed.algorithms.ddp_comm_hooks import default_hooks

        model.register_comm_hook(None, default_hooks.bf16_compress_hook)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    B = args.batch
    gen = torch.Generator().manual_seed(1234 + rank)
    host_x = torch.randn(B, 3, 224, 224, generator=gen).pin_memory()
    host_y = torch.randint(0, 1000, (B,), generator=gen).pin_memory()
    dev_x = host_x.to(device)
    dev_y = host_y.to(device)
    loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
    last = {}  # loss of the most recent timed step, for --dump-outputs

    def timed(region_steps, resident: bool):
        """Returns ms for `region_steps` steps (device time, this rank)."""
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(region_steps):
            if resident:
                x, y = dev_x, dev_y
            else:
                x = host_x.to(device, non_blocking=True)
                y = host_y.to(device, non_blocking=True)
            loss = train_step(model, opt, x, y, "cuda")
            if not resident:
                loss_host.copy_(loss.detach().float(), non_blocking=True)
        t1.record()
        torch.cuda.synchronize()
        last["loss"] = loss
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1)

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # CPU tensor -> gloo side of the group
        return float(t.item())

    log("warm-up")
    for _ in range(max(args.warmup, 3)):
        train_step(model, opt, dev_x, dev_y, "cuda")
    torch.cuda.synchronize()
    log(f"timing {args.steps} steps (inputs resident in HBM)")

    launches0 = pg.comm.launch_count if (pg is not None and pg.comm is not None) else 0
    if pg is not None:
        pg.timings = []
        pg.record_timings = True
    with ClockSampler(local_rank) as clocks:
        ms = max_over_ranks(timed(args.steps, resident=True))
    if pg is not None:
        pg.record_timings = False
    launches = (pg.comm.launch_count - launches0) if (pg is not None and pg.comm is not None) else 0
    kernel_ms = []
    kernel_bytes = []
    if pg is not None:
        # only the fused gradient-bucket launches ("grad"); DDP's per-forward buffer broadcasts and
        # anything else that goes through the process group are not the roofline kernel
        for start, end, nbytes, tag in pg.timings:
            if tag == "grad":
                kernel_ms.append(start.elapsed_time(end))
                kernel_bytes.append(nbytes)
    log(f"device-timed: {ms / args.steps:.2f} ms/step; timing end-to-end (host batch in, loss out)")
    # end to end: host batch in, loss out, every step
    if args.profile:
        ms_e2e = ms
    else:
        for _ in range(2):
            timed(1, resident=False)
        ms_e2e = max_over_ranks(timed(args.steps, resident=False))
    if args.dump_outputs and rank == 0:  # DDP keeps every replica identical
        dump_outputs(args.dump_outputs, model.module, last["loss"])
        log(f"outputs of the last timed step written to {args.dump_outputs}")

    global_batch = B * world
    value = global_batch * args.steps / (ms / 1e3)
    e2e_value = global_batch * args.steps / (ms_e2e / 1e3)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"

    def ncu_traffic():
        """dram__bytes_read.sum + dram__bytes_write.sum per launch of grad_local_kernel from the
        committed `ncu --set full` capture (profiles/r02/grad_local_kernel_ncu_full.csv)."""
        try:
            import csv

            rows = list(csv.reader(open(os.path.join(ROOT, "profiles", "r02", "grad_local_kernel_ncu_full.csv"))))
            hdr, units, data = rows[0], rows[1], rows[2:]
            ri, wi = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            tot = [float(d[ri]) * scale[units[ri]] + float(d[wi]) * scale[units[wi]] for d in data]
            return sum(tot) / len(tot)
        except Exception:
            return None

    roofline = None
    if kernel_ms:
        avg_ms = sum(kernel_ms) / len(kernel_ms)
        avg_elems = sum(kernel_bytes) / len(kernel_bytes) / 4.0  # fp32 elements per launch
        if world == 1:
            # local stage of the gradient path: read fp32 + write fp32 per element
            alg = avg_elems * 8.0
            roofline = {"bound": "hbm", "achieved": alg / (avg_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "traffic": ncu_traffic(), "kernel": "grad_local_kernel", "peak_source": peak_src,
                        "note": "launches overlap the backward pass (separate stream); the ncu capture shows "
                                "the fp32 write-back staying in the 126 MB L2",
                        "launch_ms": avg_ms, "algorithmic_bytes_per_launch": alg}
        else:
            wire_b = 2.0 if args.grad_wire == "bf16" else 4.0
            alg = avg_elems * wire_b * 2.0 * (world - 1) / world  # nccl-tests bus bytes
            roofline = {"bound": "nvlink", "achieved": alg / (avg_ms * 1e-3) / 1e9, "peak": 900.0, "unit": "GB/s",
                        "traffic": None, "kernel": "grad_allreduce_kernel", "launch_ms": avg_ms,
                        "peak_source": "nominal NVLink 5 per direction (measured peer copy 770 GB/s)",
                        "algorithmic_bytes_per_launch": alg,
                        "note": "in-step launches include waiting for the slowest rank's bucket"}
        roofline["frac"] = roofline["achieved"] / roofline["peak"]

    sweep = ag_sweep = parity = nccl_cmp = ppo = None
    if world > 1 and not args.no_sweep and not args.profile:
        if args.impl == "b200":
            log("parity check against the gloo side of the process group (untimed)")
            parity = parity_check(pg, rank, world, device)
        log("all-reduce / all-gather bandwidth sweeps")
        sweep = collective_sweep(args, pg, rank, world, device, "allreduce")
        ag_sweep = collective_sweep(args, pg, rank, world, device, "allgather")
        ppo = ppo_allreduce_latency(args, pg, rank, world, device)
        if args.impl == "b200" and not args.no_nccl_comparator:
            log("NCCL comparator: same sweeps and the same DDP step over a ProcessGroupNCCL (not the product)")
            # free the product's model first: the comparator builds its own
            nccl_cmp = nccl_comparator(args, rank, world, device, dev_x, dev_y, host_x, host_y, loss_host)

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "impl": args.impl,
            "config": {"workload": "ResNet-50 DDP training step (BASELINE configs[1])", "model": "resnet50",
                       "global_batch": global_batch, "per_gpu_batch": B, "image": "3x224x224",
                       "optimizer": "adam lr=1e-3", "autocast": "bf16", "parallelism": f"dp{world}",
                       "grad_sync": ("b200 fused hook wire=" + args.grad_wire) if args.impl == "b200"
                       else "torch DDP + NCCL" + (" bf16_compress_hook" if args.grad_wire == "bf16" else ""),
                       "ddp_at_world_1": world == 1,
                       "l2": "per-step activations+weights (>1 GB) exceed the 126 MB L2; no explicit flush"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int((host_x.numel() * 4 + host_y.numel() * 8) * world),
                    "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
            "model_flops_frac": value * FLOPS_PER_SAMPLE / world / (float(peaks.get("bf16_tflops_sustained", 1411.0)) * 1e12),
        }
        if roofline is not None:
            line["roofline"] = roofline
        if sweep is not None:
            line["allreduce_sweep"] = sweep
        if ag_sweep is not None:
            line["allgather_sweep"] = ag_sweep
        if ppo is not None:
            line["ppo_mlp_allreduce"] = ppo
        if parity is not None:
            line["parity_check"] = parity
        if nccl_cmp is not None:
            line["nccl_comparator"] = nccl_cmp
    if world > 1:
        dist.barrier()
    dist.destroy_process_group()
    return line


def _time_collective(one, iters, world):
    """5 warm-up + `iters` timed launches, CUDA events on the launching stream, max over ranks -> us."""
    import torch
    import torch.distributed as dist

    for _ in range(5):
        one()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        one()
    t1.record()
    torch.cuda.synchronize()
    t = torch.tensor([t0.elapsed_time(t1) / iters], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)  # CPU tensor -> gloo
    return float(t.item()) * 1e3


def collective_sweep(args, pg, rank, world, device, op, group=None):
    """Bus bandwidth vs message size, nccl-tests convention (SURVEY 8d):
      allreduce: S = tensor bytes, busbw = S/t * 2(n-1)/n, in place on an ordinary fp32 tensor;
      allgather: S = total gathered bytes (n x per-rank), busbw = S/t * (n-1)/n.
    `group` = a torch ProcessGroup to time instead of the product (the NCCL comparator)."""
    import torch
    import torch.distributed as dist

    out = []
    sizes = [1 << s for s in range(10, 31, 2)]  # 1 KiB .. 1 GiB
    for nbytes in sizes:
        iters = 20 if nbytes <= (256 << 20) else 8
        if op == "allreduce":
            x = torch.ones(nbytes // 4, device=device)
            if group is None and args.impl == "b200":
                one = lambda: pg.comm.allreduce(x)  # noqa: E731
            else:
                one = lambda: dist.all_reduce(x, group=group)  # noqa: E731
            factor = 2 * (world - 1) / world
            bufs = (x,)
        else:
            per = max(nbytes // world // 4, 1)
            x = torch.ones(per, device=device)
            y = torch.empty(per * world, device=device)
            if group is None and args.impl == "b200":
                one = lambda: pg.comm.allgather_into(y, x)  # noqa: E731
            else:
                one = lambda: dist.all_gather_into_tensor(y, x, group=group)  # noqa: E731
            factor = (world - 1) / world
            nbytes = per * world * 4
            bufs = (x, y)
        us = _time_collective(one, iters, world)
        algbw = nbytes / (us * 1e-6) / 1e9
        out.append({"bytes": nbytes, "us": round(us, 2), "algbw_gbs": round(algbw, 2), "busbw_gbs": round(algbw * factor, 2)})
        del bufs, x
    return out


def ppo_mlp_numel():
    """RLlib's default PPO module (rllib/core/rl_module/default_model_config.py:65-69: two 256-wide
    tanh layers, separate policy and value networks) on a CartPole-sized space (4 observations,
    2 actions): the gradient vector a 4-learner LearnerGroup all-reduces every update
    (BASELINE.json configs[3])."""
    import torch.nn as nn

    def mlp(out):
        return nn.Sequential(nn.Linear(4, 256), nn.Tanh(), nn.Linear(256, 256), nn.Tanh(), nn.Linear(256, out))

    return sum(p.numel() for m in (mlp(2), mlp(1)) for p in m.parameters())


def ppo_allreduce_latency(args, pg, rank, world, device, group=None):
    import torch
    import torch.distributed as dist

    numel = ppo_mlp_numel()
    g = torch.ones(numel, device=device)
    if group is None and args.impl == "b200":
        one = lambda: pg.comm.allreduce(g)  # noqa: E731
    else:
        one = lambda: dist.all_reduce(g, group=group)  # noqa: E731
    us = _time_collective(one, 200, world)
    return {"numel": numel, "bytes": numel * 4, "us_per_allreduce": round(us, 2), "world": world,
            "note": "fp32 gradient vector of RLlib's default PPO MLPs; BASELINE configs[3] is world 4"}


def parity_check(pg, rank, world, device):
    """Multi-GPU parity where the driver can see it: seeded inputs through the product kernels
    (AUTO algorithm selection: NVLS / pipelined / staged as the size dictates), compared with the
    gloo side of the SAME process group (the reference's CPU backend, torch_gloo_collective_group.py:
    208-290) -- fp32 within 1e-6 * sum_r|x_r| (north_star), integers and copies bit exact, every
    replica bit-identical.  Raises on the first mismatch; returns the summary for the JSON line."""
    import torch
    import torch.distributed as dist

    comm = pg.comm
    cases = failed = 0
    max_rel = 0.0
    detail = []

    def seeded(numel, dtype, r, salt=0):
        gen = torch.Generator().manual_seed(1234 + r + 1000 * salt)
        if dtype.is_floating_point:
            return torch.randn(numel, generator=gen).to(dtype)
        return torch.randint(-1000, 1000, (numel,), generator=gen, dtype=dtype)

    def replicas_identical(t):
        v = t.view(torch.uint8).view(-1)
        pad = (-v.numel()) % 8
        if pad:
            v = torch.cat([v, torch.zeros(pad, dtype=torch.uint8, device=v.device)])
        w = v.view(torch.int64)
        sig = torch.stack([w.sum(), (w ^ (w >> 7)).sum()]).cpu()
        sigs = [torch.zeros_like(sig) for _ in range(world)]
        dist.all_gather(sigs, sig)  # CPU -> gloo
        return all(torch.equal(x, sigs[0]) for x in sigs)

    def record(name, ok, rel=0.0):
        nonlocal cases, failed, max_rel
        cases += 1
        max_rel = max(max_rel, float(rel))
        if not ok:
            failed += 1
        detail.append({"case": name, "ok": bool(ok), "max_rel": float(rel)})

    MiB = 1 << 20
    # ---- all-reduce fp32 / bf16 / int32 ------------------------------------------------------
    for dtype, sizes, tol in ((torch.float32, (1 * MiB, 64 * MiB, 256 * MiB), 1e-6), (torch.bfloat16, (1 * MiB, 64 * MiB), 2.0 ** -6),
                              (torch.int32, (1 * MiB, 64 * MiB), 0.0)):
        for nbytes in sizes:
            numel = nbytes // torch.empty((), dtype=dtype).element_size()
            host = seeded(numel, dtype, rank)
            x = host.to(device)
            comm.allreduce(x)
            torch.cuda.synchronize()
            got = x.cpu()
            if dtype == torch.int32:
                ref = host.clone()
                dist.all_reduce(ref)  # gloo
                ok = torch.equal(got, ref)
                rel = 0.0
            else:
                sabs = host.float().abs()
                dist.all_reduce(sabs)
                ref = host.float().clone()  # .float() of an fp32 tensor is the tensor itself
                dist.all_reduce(ref)
                err = (got.float() - (ref if dtype == torch.float32 else ref.to(dtype).float())).abs()
                rel = float((err / sabs.clamp_min(1e-30)).max())
                ok = bool((err <= tol * sabs + 1e-30).all())
            ok = ok and replicas_identical(x)
            record(f"allreduce/{str(dtype)[6:]}/{nbytes >> 20}MiB", ok, rel)
            del x, got, ref
    # ---- fused gradient kernel (fp32 bucket, bf16 wire, scale 1/world) ------------------------
    numel = 25 * MiB // 4
    host = seeded(numel, torch.float32, rank, salt=1)
    gbuf = host.to(device)
    comm.grad_allreduce(gbuf, 1.0 / world, torch.bfloat16)
    torch.cuda.synchronize()
    wire = (host * (1.0 / world)).to(torch.bfloat16).float()
    sabs = wire.abs()
    dist.all_reduce(sabs)
    ref = wire.clone()
    dist.all_reduce(ref)
    err = (gbuf.cpu() - ref.to(torch.bfloat16).float()).abs()
    rel = float((err / sabs.clamp_min(1e-30)).max())
    record("grad_allreduce/bf16wire/25MiB", bool((err <= 2.0 ** -6 * sabs + 1e-30).all()) and replicas_identical(gbuf), rel)
    del gbuf
    # ---- all-gather, reduce-scatter, broadcast (64 MiB total / per op) ------------------------
    per = 64 * MiB // 4 // world
    x = seeded(per, torch.float32, rank, salt=2).to(device)
    y = torch.empty(per * world, device=device)
    comm.allgather_into(y, x)
    torch.cuda.synchronize()
    want = torch.cat([seeded(per, torch.float32, p, salt=2) for p in range(world)])
    record("allgather/f32/64MiB", torch.equal(y.cpu(), want))
    full = seeded(per * world, torch.float32, rank, salt=3)
    out = torch.empty(per, device=device)
    comm.reducescatter_from(out, full.to(device))
    torch.cuda.synchronize()
    sabs = full.abs()
    dist.all_reduce(sabs)
    ref = full.clone()
    dist.all_reduce(ref)  # the reference's gloo reducescatter is n all-reduces (torch_gloo_collective_group.py:260-282)
    sl = slice(rank * per, (rank + 1) * per)
    err = (out.cpu() - ref[sl]).abs()
    rel = float((err / sabs[sl].clamp_min(1e-30)).max())
    record("reducescatter/f32/64MiB", bool((err <= 1e-6 * sabs[sl] + 1e-30).all()), rel)
    root = world - 1
    b = seeded(16 * MiB // 4, torch.float32, rank, salt=4).to(device)
    comm.broadcast(b, root)
    torch.cuda.synchronize()
    record("broadcast/f32/16MiB", torch.equal(b.cpu(), seeded(16 * MiB // 4, torch.float32, root, salt=4)))
    # every rank must agree that nothing failed
    flag = torch.tensor([failed], dtype=torch.int64)
    dist.all_reduce(flag)
    summary = {"cases": cases, "failed": int(flag.item()), "max_rel": max_rel, "multicast": bool(comm.has_multicast),
               "tolerance": "fp32 1e-6*sum|x_r| vs gloo; bf16 2^-6*sum|x_r| (the NVSwitch rounds partial sums in bf16: up to n-1 roundings of 2^-9); int/copies bit exact; "
                            "replicas bit-identical", "detail": detail}
    if summary["failed"]:
        raise RuntimeError(f"parity check failed: {json.dumps(summary)}")
    return summary


def nccl_comparator(args, rank, world, device, dev_x, dev_y, host_x, host_y, loss_host):
    """The reference's GPU backend is NCCL (nccl_collective_group.py / torch c10d); the reference
    itself cannot run here (no Ray, no cupy), so the comparator is torch's ProcessGroupNCCL on the
    same box, in the same processes: the same sweeps and the same DDP step with bf16_compress_hook."""
    import torch
    import torch.distributed as dist
    from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
    from torch.nn.parallel import DistributedDataParallel as DDP

    nccl = dist.new_group(backend="nccl")
    fake_args = argparse.Namespace(impl="nccl")
    out = {"backend": f"torch ProcessGroupNCCL, NCCL {'.'.join(map(str, torch.cuda.nccl.version()))}",
           "allreduce_sweep": collective_sweep(fake_args, None, rank, world, device, "allreduce", group=nccl),
           "allgather_sweep": collective_sweep(fake_args, None, rank, world, device, "allgather", group=nccl),
           "ppo_mlp_allreduce": ppo_allreduce_latency(fake_args, None, rank, world, device, group=nccl)}
    model = DDP(build(device), device_ids=[device], output_device=device, process_group=nccl)
    if args.grad_wire == "bf16":
        model.register_comm_hook(nccl, default_hooks.bf16_compress_hook)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)

    def timed(steps, resident):
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            if resident:
                x, y = dev_x, dev_y
            else:
                x = host_x.to(device, non_blocking=True)
                y = host_y.to(device, non_blocking=True)
            loss = train_step(model, opt, x, y, "cuda")
            if not resident:
                loss_host.copy_(loss.detach().float(), non_blocking=True)
        t1.record()
        torch.cuda.synchronize()
        t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 5)):  # NCCL connects lazily and autotunes in its first steps
        train_step(model, opt, dev_x, dev_y, "cuda")
    timed(2, False)
    B = dev_x.shape[0]
    ms = timed(args.steps, True)
    ms_e2e = timed(args.steps, False)
    out["samples_s"] = B * world * args.steps / (ms / 1e3)
    out["e2e_samples_s"] = B * world * args.steps / (ms_e2e / 1e3)
    out["ms_per_step"] = ms / args.steps
    out["grad_sync"] = "torch DDP + NCCL" + (" bf16_compress_hook" if args.grad_wire == "bf16" else "")
    del model, opt
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_worker(spec_path):
    """One gloo rank of the reference's CPU path: TorchTrainer(use_gpu=False) == torch DDP over
    gloo (python/ray/train/torch/config.py:186-196 picks gloo without GPUs)."""
    import torch
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP

    spec = json.load(open(spec_path))
    rank, world = int(os.environ["RANK"]), spec["world"]
    torch.set_num_threads(max(1, spec["threads"]))
    dist.init_process_group("gloo", init_method=f"file://{spec['init']}", rank=rank, world_size=world)
    model = build(torch.device("cpu"))
    if world > 1:
        model = DDP(model)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    B = spec["batch"]
    gen = torch.Generator().manual_seed(1234 + rank)
    x = torch.randn(B, 3, 224, 224, generator=gen)
    y = torch.randint(0, 1000, (B,), generator=gen)
    for _ in range(spec["warmup"]):
        train_step(model, opt, x, y, "cpu")
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(spec["steps"]):
        train_step(model, opt, x, y, "cpu")
    dist.barrier()
    dt = time.perf_counter() - t0
    if rank == 0:
        json.dump({"seconds": dt}, open(spec["out"], "w"))
    dist.destroy_process_group()


def run_cpu_reference(world, steps, warmup, batch):
    """Runs the CPU path on this host's cores; returns (samples/s, threads used, seconds)."""
    cores = len(os.sched_getaffinity(0))
    with tempfile.TemporaryDirectory(prefix="b200_cpu_ref_") as d:
        spec = {"world": world, "threads": max(1, min(cores // world, 32)), "batch": batch, "steps": steps,
                "warmup": warmup, "init": os.path.join(d, "rdzv"), "out": os.path.join(d, "out.json")}
        path = os.path.join(d, "spec.json")
        json.dump(spec, open(path, "w"))
        procs = []
        for r in range(world):
            env = dict(os.environ, RANK=str(r), OMP_NUM_THREADS=str(spec["threads"]), CUDA_VISIBLE_DEVICES="")
            procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), "--cpu-worker", path], env=env))
        deadline = time.time() + 600
        for p in procs:
            try:
                p.wait(timeout=max(1.0, deadline - time.time()))
            except subprocess.TimeoutExpired:
                for q in procs:
                    q.kill()
                raise RuntimeError("CPU reference worker timed out")
        if any(p.returncode for p in procs):
            raise RuntimeError("CPU reference worker failed")
        secs = json.load(open(spec["out"]))["seconds"]
    return world * batch * steps / secs, world * spec["threads"], secs


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (gloo DDP) on the
    box's host cores, every step a bounded sample (small per-worker batch) of the workload."""
    rank, _, world_env = env_rank()
    if rank != 0:
        return None
    world = max(args.gpus, 1)
    batch = 4
    value, cores, secs = run_cpu_reference(world, args.steps, max(args.warmup, 1), batch)
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "impl": "reference",
        "config": {"workload": "ResNet-50 DDP training step (BASELINE configs[1])", "model": "resnet50",
                   "global_batch": batch * world, "per_gpu_batch": batch, "parallelism": f"dp{world}",
                   "grad_sync": "torch DDP + gloo (the reference's CPU backend)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": f"{args.steps} steps x {world} gloo workers x batch {batch} on host cores"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main():
    import faulthandler

    faulthandler.dump_traceback_later(int(os.environ.get("B200_BENCH_WATCHDOG_S", "1500")), exit=True)
    args = parse_args()
    if args.cpu_worker:
        cpu_worker(args.cpu_worker)
        return
    if args.impl == "reference":
        line = run_reference(args)
    else:
        line = run_gpu(args)
        if line is not None and line["n_gpus"] == 1 and not args.no_cpu_baseline and args.impl == "b200":
            try:
                log("cpu_baseline: reference CPU path on the host cores (bounded sample)")
                v, cores, secs = run_cpu_reference(1, 6, 1, 4)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference",
                                        "sample": f"6 steps, batch 4, 1 worker, {secs:.1f}s of host time "
                                                  "(torch CPU ResNet-50 + DDP/gloo path)"}
            except Exception as exc:  # the GPU numbers stand on their own
                line["cpu_baseline"] = {"error": str(exc)}
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
