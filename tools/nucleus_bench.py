"""Nucleus (top-p) summarisation timings on one GPU: what the cut costs inside the sampled roll-out launch.

    python tools/nucleus_bench.py [--out profiles/r07_nucleus_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/sample_bench.py (synthetic, seeded, four rotating batches of one padded-shape bucket):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 steps
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 steps
On batch 0's encoder outputs, CUDA events, medians after a warm-up:
  N{n}_k{k}_p{p}   MultimodalAttentionDecoder.sample (one launch); p1 is the plain sampled roll-out, the reference arm.
                   cfg3: N in 1, 4, 16 at top_k 0 with top_p 1, 0.5, 0.9, and top_k 8 with top_p 1, 0.9; cfg5: N in 1, 4 at top_k 0
                   with top_p 1, 0.9
  N4_k0_p0.9_constrained   the same with no_repeat=True, min_sentences=3
  N4_host_loop_p0.9        (cfg3) the same 4 samples as a Python loop of the fused step kernel at B N rows and
                           mmb_sample_pick_nucleus per step
and at config-3 shapes the Summarizer replay + Summary.to_lists per batch for N = 4, top_p 0.9 (host clock, ends in the host copy).
Writes one JSON file with the GPU's name, power limit and max SM clock beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from sample_bench import replicated  # noqa: E402
from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, N_ROTATE, WORKLOADS, event_time, gpu_info, host_time, stats  # noqa: E402

ARMS = {"cfg3": [(n, 0, p) for n in (1, 4, 16) for p in (1.0, 0.5, 0.9)] + [(n, 8, p) for n in (1, 4, 16) for p in (1.0, 0.9)],
        "cfg5": [(n, 0, p) for n in (1, 4) for p in (1.0, 0.9)]}


def host_loop(dec, emb, h0, enc_a, enc_i, mask, S, N, key, top_p):
    """N samples per video as a Python loop: the fused step kernel over B N rows (the B-video tensors replicated), then the pick."""
    from mmbidaf_b200 import ops
    rs = replicated(dec, enc_a, enc_i, N)
    B, Lt, H = rs.B // N, rs.Lt, rs.H
    R, dev = B * N, emb.device
    emb_r, mask_r = emb.repeat_interleave(N, 0), ops._u8(mask.bool().repeat_interleave(N, 0))
    base = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(N)
    rows = torch.arange(R, device=dev)
    sent, h = emb.new_zeros(R, emb.shape[2]), h0.reshape(B, H).repeat_interleave(N, 0).contiguous()
    cell, cov = torch.zeros(R, H, device=dev), torch.zeros(R, Lt, device=dev)
    for s in range(S):
        p, h, cell, _, cov, *_ = ops.decoder_step_fwd(rs, sent.contiguous(), h, cell, cov, mask_r)
        sent = emb_r[rows, ops.sample_pick(p, key, base, S, s, N, top_p=top_p).clamp(0, Lt - 1)]


def run_workload(name, iters):
    from mmbidaf_b200 import ops
    from mmbidaf_b200.layers.encoding import length_plan
    from mmbidaf_b200.models import MMBiDAF
    from mmbidaf_b200.summarize import Summarizer
    from mmbidaf_b200.synth import make_batch
    c = WORKLOADS[name]
    dev = torch.device("cuda")
    torch.manual_seed(224)
    model = MMBiDAF(HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, dev, drop_prob=0.2, max_transcript_length=c["m"]).to(dev)
    model.eval()
    batches = [make_batch(c["batch"], c["lt"], c["la"], c["li"], c["steps"], E_TEXT, E_AUDIO, E_IMAGE, seed=224 + i).to(dev)
               for i in range(N_ROTATE)]
    S = c["steps"]
    res = {"workload": name, "shape": c, "rotating_batches": N_ROTATE, "arms": {}}
    b = batches[0]
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    lens = length_plan(b.text_len, dev).len_i32.clone()
    key = ops.seed_key(224, dev)

    def timed(k, fn):
        for _ in range(3):
            fn()
        res["arms"][k] = stats(event_time(fn, iters))
        print(name, k, res["arms"][k]["median_ms"], flush=True)

    for N, top_k, top_p in ARMS[name]:
        timed(f"N{N}_k{top_k}_p{top_p:g}", lambda: dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, N, key, 1.0, top_k, top_p=top_p))
    timed("N4_k0_p0.9_constrained", lambda: dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, 4, key, 1.0, 0, True, 3, top_p=0.9))
    if name == "cfg3":
        saved = os.environ.get("MMB_DECODER_CUT")
        os.environ["MMB_DECODER_CUT"] = "fused"
        try:
            with torch.no_grad():
                timed("N4_host_loop_p0.9", lambda: host_loop(dec, b.text, h0, enc_a, enc_i, mask, S, 4, key, 0.9))
        finally:
            if saved is None:
                os.environ.pop("MMB_DECODER_CUT", None)
            else:
                os.environ["MMB_DECODER_CUT"] = saved
        summarizer = Summarizer(model)
        fn = lambda bb: summarizer(bb, num_samples=4, top_p=0.9).to_lists()                         # noqa: E731
        for bb in batches:
            fn(bb)
        res["arms"]["N4_p0.9_summarizer"] = stats(host_time(fn, batches, iters))
        print(name, "N4_p0.9_summarizer", res["arms"]["N4_p0.9_summarizer"]["median_ms"], flush=True)
        model.eval()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_nucleus_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nucleus_bench: needs a CUDA device (no CPU timing)")
    import mmbidaf_b200
    mmbidaf_b200.set_precision(args.precision)
    out = {"gpu": gpu_info(), "precision": args.precision, "iters": args.iters, "workloads": []}
    for name in ([args.only] if args.only else list(WORKLOADS)):
        out["workloads"].append(run_workload(name, args.iters))
        print(json.dumps(out["workloads"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
