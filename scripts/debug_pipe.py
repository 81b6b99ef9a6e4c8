"""Debug helper: run the pipelined all-reduce variants and describe any mismatch."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from ray_b200 import _native as N
from ray_b200.testing import LocalGroup

world = int(sys.argv[1]) if len(sys.argv) > 1 else 2
g = LocalGroup(world, timeout_ms=10000, staging_bytes=40 << 20, inbox_bytes=2 << 20)
print("multicast", g.has_multicast, "devices", g.devices)
MiB = 1 << 20
variants = [("peer", 2)] + ([("pull", 3)] if world == 2 else []) + ([("nvls", 1)] if g.has_multicast else [])
for vname, v in variants:
    for c in g.comms:
        c.set_param(N.PARAM_PIPE_VARIANT, v)
    for nbytes in [16, 32, 4096, 16 * 1023, 32 << 10, (32 << 10) + 16, MiB, MiB + 16, 3 * MiB + 16 * 77, 5 * MiB]:
        for rep in range(3):
            numel = nbytes // 4
            host = [(torch.randn(numel, generator=torch.Generator().manual_seed(r + rep)) * 4).round() for r in range(world)]
            xs = [h.to(g.device(r)) for r, h in enumerate(host)]
            try:
                g.run(lambda c, r: c.allreduce(xs[r], N.SUM, algo=N.ALGO_PIPE))
            except Exception as e:  # noqa: BLE001
                print(vname, nbytes, "EXC", e)
                raise
            want = torch.stack(host).sum(0)
            for r in range(world):
                got = xs[r].cpu()
                bad = (got != want).nonzero().flatten()
                if len(bad):
                    i = int(bad[0])
                    kinds = {}
                    for b in bad.tolist()[:100000]:
                        gv = float(got[b])
                        kind = "other"
                        for q in range(world):
                            if gv == float(host[q][b]):
                                kind = f"=in{q}"
                        kinds[kind] = kinds.get(kind, 0) + 1
                    print(f"{vname} {nbytes}B rep{rep} rank{r}: {len(bad)} bad of {numel}; first {i} last {int(bad[-1])} "
                          f"got {float(got[i])} want {float(want[i])} ins {[float(h[i]) for h in host]} kinds {kinds}")
        print(vname, nbytes, "done", flush=True)
g.destroy()
