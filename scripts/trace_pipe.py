"""Timeline of one pipelined all-reduce launch from the in-kernel event trace.

    python scripts/trace_pipe.py --world 2 --variant pull --mib 64
"""
import argparse
import os
import sys
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from ray_b200 import _native as N
from ray_b200.testing import LocalGroup

ap = argparse.ArgumentParser()
ap.add_argument("--world", type=int, default=2)
ap.add_argument("--variant", default="pull")
ap.add_argument("--mib", type=int, default=64)
ap.add_argument("--copy", type=int, default=-1)
ap.add_argument("--red", type=int, default=-1)
ap.add_argument("--chunk", type=int, default=-1)
ap.add_argument("--ctas", default="0,1,16,17")
args = ap.parse_args()
V = {"nvls": 1, "peer": 2, "pull": 3}[args.variant]
g = LocalGroup(args.world, timeout_ms=10000, staging_bytes=256 << 20, inbox_bytes=8 << 20)
for c in g.comms:
    c.set_param(N.PARAM_PIPE_VARIANT, V)
    c.set_param(N.PARAM_PIPE_COPY_CTAS, args.copy)
    c.set_param(N.PARAM_PIPE_RED_CTAS, args.red)
    c.set_param(N.PARAM_PIPE_CHUNK_BYTES, args.chunk << 20 if args.chunk > 0 else -1)
numel = (args.mib << 20) // 4
xs = [torch.ones(numel, device=g.device(r)) for r in range(args.world)]
for _ in range(3):
    g.run(lambda c, r: c.allreduce(xs[r], N.SUM, algo=N.ALGO_PIPE))
g.comms[0].trace_enable(1 << 20)
g.run(lambda c, r: c.allreduce(xs[r], N.SUM, algo=N.ALGO_PIPE))
ev = g.comms[0].trace_read()
ev.sort()
t0 = ev[0][0]
print(f"# {args.variant} world={args.world} {args.mib} MiB: {len(ev)} events, span {(ev[-1][0] - t0) / 1e3:.1f} us")
by_cta = defaultdict(list)
for ns, cta, e, a in ev:
    by_cta[cta].append(((ns - t0) / 1e3, e, a))
names = {1: "load", 2: "store", 3: "ringok", 4: "done<", 5: "drain", 6: "gateok", 9: "flag:see", 10: "flag:proxyfenced", 13: "flag:sysfenced", 11: "flag:arrived", 12: "flag:signal",
         30: "pl:load", 31: "pl:gatewait", 32: "pl:gateok", 33: "pl:landed", 23: "red:arrived", 41: "o:load", 42: "o:store", 43: "o:ringok", 44: "o:done<",
         45: "o:drain", 46: "o:gateok"}
for cta in [int(x) for x in args.ctas.split(",")]:
    rows = by_cta.get(cta, [])
    print(f"## CTA {cta}: {len(rows)} events")
    line = []
    for t, e, a in rows[:90]:
        line.append(f"{t:7.1f} {names.get(e, e)}({a})")
    for i in range(0, len(line), 6):
        print("   " + " | ".join(line[i:i + 6]))
# per-event-type last timestamps per role
last = defaultdict(float)
first = {}
for ns, cta, e, a in ev:
    t = (ns - t0) / 1e3
    last[e] = max(last[e], t)
    first.setdefault(e, t)
print("## first/last per event:", {names.get(e, e): (round(first[e], 1), round(last[e], 1)) for e in sorted(last)})
g.destroy()
