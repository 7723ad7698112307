"""Per-item timeline of the persistent forward (csrc/bidaf_fwd_tc5.cu), debugging aid.
    python tools/bidaf_fwd_items.py [B Lc Lq]
Per item: [0] published by the scheduler, [1] epilogue start (accumulator complete), [2] epilogue end, [3] kind, [4] SM, [5] tiles,
[7] X tile in shared memory (the MMA warp starts the item)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
B, Lc, Lq = (int(v) for v in sys.argv[1:4]) if len(sys.argv) >= 4 else (64, 512, 256)
d = 200
dev = "cuda"
nq, nc = (Lq + 127) // 128, (Lc + 127) // 128
n_items = B * (nq + 2 * nc)
trace = torch.zeros(n_items, 8, dtype=torch.int64, device=dev)
os.environ["MMB_BIDAF_FWD_ITEM_TRACE"] = str(trace.data_ptr())       # read once, at the first launch
from mmbidaf_b200 import ops  # noqa: E402

gen = torch.Generator().manual_seed(224)
c = torch.randn(B, Lc, d, generator=gen).to(dev)
q = torch.randn(B, Lq, d, generator=gen).to(dev)
cm = (torch.arange(Lc).unsqueeze(0) < torch.randint(Lc // 2, Lc + 1, (B, 1), generator=gen)).to(dev)
qm = (torch.arange(Lq).unsqueeze(0) < torch.randint(Lq // 2, Lq + 1, (B, 1), generator=gen)).to(dev)
w = [torch.randn(d, generator=gen).to(dev) * 0.1 for _ in range(3)]
bias = torch.zeros(1, device=dev)
for _ in range(4):
    ops.bidaf_fwd(c, q, cm, qm, w[0], w[1], w[2], bias, None, None, 1.0, 1)
torch.cuda.synchronize()
t = trace.cpu()
t0 = int(t[:, 0].min())
print(f"{n_items} items; span {int(t[:, 2].max()) - t0} ns on {len(set(t[:, 4].tolist()))} SMs")
for kind, name in enumerate(("Q2C", "C2QA", "C2QB")):
    x = t[t[:, 3] == kind]
    if not len(x):
        continue
    print(f"{name}: {len(x)} items, tiles {x[:, 5].float().mean():.1f}; published {int(x[:, 0].min()) - t0}..{int(x[:, 0].max()) - t0} ns; "
          f"publish -> accumulator complete {(x[:, 1] - x[:, 0]).float().mean():.0f} ns; epilogue {(x[:, 2] - x[:, 1]).float().mean():.0f} ns "
          f"(max {int((x[:, 2] - x[:, 1]).max())})")
# per SM: items in order of publication; loop time of an item ~ difference between consecutive 'accumulator complete' stamps
per_tile = []
for smid in sorted(set(t[:, 4].tolist()))[:4]:
    x = t[t[:, 4] == smid]
    x = x[x[:, 0].argsort()]
    print(f"SM {smid}: " + "  ".join(f"{('Q', 'A', 'B')[int(r[3])]}{int(r[5])}t pub {int(r[0]) - t0}" + (f" mma {int(r[7]) - t0}" if int(r[7]) else "")
                                     + f" acc {int(r[1]) - t0} end {int(r[2]) - t0}" for r in x))
for smid in set(t[:, 4].tolist()):
    x = t[t[:, 4] == smid]
    x = x[x[:, 1].argsort()]
    for i in range(1, len(x)):
        per_tile.append(float(x[i, 1] - x[i - 1, 1]) / max(int(x[i, 5]), 1))
if per_tile:
    pt = torch.tensor(per_tile)
    print(f"accumulator-complete to accumulator-complete per tile: mean {pt.mean():.0f} ns, median {pt.median():.0f} ns (64-column tiles)")
