"""Event log of CTA 0 of the persistent forward (csrc/bidaf_fwd_tc5.cu), debugging aid: per role a list of (code, clock64).
    python tools/bidaf_fwd_events.py [B Lc Lq]
MMA warp: kind (0 Q, 1 A, 2 B) pass taken, 10 X tile there, 200+t Y tile there, 300+t S buffer free -> S(t) issued, 400+t P(t) there -> P V(t) issued.
Soft-max warp 0: 200+t S(t) there, 300+t S(t) in registers, 400+t P computed, 500+t P buffer free, 600+t P(t) written.
TMA warp: kind published, 100+t slot free -> Y tile t requested."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
B, Lc, Lq = (int(v) for v in sys.argv[1:4]) if len(sys.argv) >= 4 else (64, 512, 256)
d = 200
dev = "cuda"
ev = torch.zeros(4, 2048, dtype=torch.int64, device=dev)
os.environ["MMB_BIDAF_FWD_EV_TRACE"] = str(ev.data_ptr())
from mmbidaf_b200 import ops  # noqa: E402

gen = torch.Generator().manual_seed(224)
c = torch.randn(B, Lc, d, generator=gen).to(dev)
q = torch.randn(B, Lq, d, generator=gen).to(dev)
cm = (torch.arange(Lc).unsqueeze(0) < torch.randint(Lc // 2, Lc + 1, (B, 1), generator=gen)).to(dev)
qm = (torch.arange(Lq).unsqueeze(0) < torch.randint(Lq // 2, Lq + 1, (B, 1), generator=gen)).to(dev)
w = [torch.randn(d, generator=gen).to(dev) * 0.1 for _ in range(3)]
bias = torch.zeros(1, device=dev)
for _ in range(3):
    ev.zero_()
    ops.bidaf_fwd(c, q, cm, qm, w[0], w[1], w[2], bias, None, None, 1.0, 1)
torch.cuda.synchronize()
e = ev.cpu().view(4, 1024, 2)
t0 = min(int(e[r, 0, 1]) for r in range(4) if int(e[r, 0, 1]))
for r, name in enumerate(("mma", "softmax0", "tma", "epilogue0")):
    rows = [(int(c_), int(t_) - t0) for c_, t_ in e[r].tolist() if t_]
    print(name + ": " + " ".join(f"{c_}@{t_}" for c_, t_ in rows[:160]))
