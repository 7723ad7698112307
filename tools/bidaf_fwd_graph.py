"""Graph-replayed timing of the fused BiDAF forward (bf16 tier) at BASELINE config 2, plus a check of its output against the
fp32 tier on the same inputs.  The four calls over four rotating input sets are captured into one CUDA graph (a call from Python
costs ~40 us of host time, more than the kernels).
    python tools/bidaf_fwd_graph.py [--shape B Lc Lq] [--rounds 20]
"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mmbidaf_b200 import ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--shape", type=int, nargs=3, default=[64, 512, 256])
ap.add_argument("--rounds", type=int, default=20)
ap.add_argument("--no-check", action="store_true")
a = ap.parse_args()
B, Lc, Lq = a.shape
d = 200
dev = torch.device("cuda")
gen = torch.Generator().manual_seed(224)
sets = []
for _ in range(4):
    c = torch.randn(B, Lc, d, generator=gen).to(dev)
    q = torch.randn(B, Lq, d, generator=gen).to(dev)
    cm = (torch.arange(Lc).unsqueeze(0) < torch.randint(Lc // 2, Lc + 1, (B, 1), generator=gen)).to(dev)
    qm = (torch.arange(Lq).unsqueeze(0) < torch.randint(Lq // 2, Lq + 1, (B, 1), generator=gen)).to(dev)
    sets.append((c, q, cm, qm))
w = [torch.randn(d, generator=gen).to(dev) * 0.1 for _ in range(3)]
bias = torch.full((1,), 0.3, device=dev)
run = lambda s, prec, aux=True: ops.bidaf_fwd(s[0], s[1], s[2], s[3], w[0], w[1], w[2], bias, precision=prec, aux=aux)
if not a.no_check:
    s = sets[0]
    got = run(s, ops.PREC_BF16)
    want = run(s, ops.PREC_FP32)
    torch.cuda.synchronize()
    for name, g, r in zip(("out", "q2c", "lse_row", "lse_col"), got, want):
        err = float((g - r).abs().max()) / max(float(r.abs().max()), 1e-30)
        print(f"  {name}: max|d|/max|ref| = {err:.3e}{'' if torch.isfinite(g).all() else '  NON-FINITE'}")
side = torch.cuda.Stream(dev)
side.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(side):
    for i in range(4):
        run(sets[i], ops.PREC_BF16, False)
torch.cuda.current_stream().wait_stream(side)
torch.cuda.synchronize()
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph):
    keep = [run(s, ops.PREC_BF16, False) for s in sets]                   # as bench.py: the inference path (only out)
for _ in range(3):
    graph.replay()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.synchronize()
e0.record()
for _ in range(a.rounds):
    graph.replay()
e1.record()
torch.cuda.synchronize()
t = e0.elapsed_time(e1) / a.rounds / 4 * 1e3
algo = 4 * B * (Lc * d + Lq * d + Lc * 4 * d) + B * (Lc + Lq)
print(f"B={B} Lc={Lc} Lq={Lq}: {t:.1f} us/forward (graph replay), "
      f"{algo / t / 1e3:.1f} GB/s algorithmic ({algo / t / 1e3 / 6553.3 * 100:.1f}% of 6553 GB/s)")
