"""Sequence-level training timings on one GPU: the differentiable scores of N candidates per video, forward + backward.

    python tools/sequence_scores_bench.py [--out profiles/r10_sequence_scores_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/summarize_bench.py (synthetic, seeded): cfg3 (B=32, Lt 409, M 409, 12 steps; N in 1, 4, 16) and cfg5 (B=16,
Lt=4096, M=4096, 16 steps; N in 1, 4).  On batch 0's encoder outputs (leaves that require grad), the candidates N sampled summaries
per video, CUDA events, median and min after a warm-up of 3 calls:
  N{n}_forced_train    MultimodalAttentionDecoder.force_train + backward: one launch forward, one launch backward (B N clusters)
  N{n}_step_autograd   the hand-written alternative: MultimodalAttentionDecoder.step under autograd over the B N rows (the encoder
                       outputs repeated N times), then its backward, on the cut ops.decoder_cut picks (the five-kernel chunk cut
                       when B N Lt > 20000, else one cluster kernel per step)
  N{n}_step_autograd_fused  the same with MMB_DECODER_CUT=fused: one cluster kernel per step forward and backward at every size, the
                       per-step counterpart of the two roll-outs
  N{n}_sequence_scores the whole MMBiDAF.sequence_scores in training mode + backward of (logp + loss).sum()
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

from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, WORKLOADS, event_time, gpu_info, stats  # noqa: E402

ARMS = {"cfg3": (1, 4, 16), "cfg5": (1, 4)}


def step_autograd(dec, emb, h0, enc_a, enc_i, mask, tokens):
    """The forced roll-out written by hand: ``dec.step`` under autograd over the B N rows, then the backward of its loss terms."""
    B, N, S = tokens.shape
    R, Lt = B * N, emb.shape[1]
    ea, ei = enc_a.repeat_interleave(N, 0), enc_i.repeat_interleave(N, 0)
    emb_r, mask_r = emb.repeat_interleave(N, 0), mask.repeat_interleave(N, 0)
    rows, tok = torch.arange(R, device=emb.device), tokens.reshape(R, S)
    sent = emb.new_zeros(R, 1, emb.shape[2])
    h = h0.reshape(B, 1, -1).repeat_interleave(N, 0)
    cell, cov = emb.new_zeros(1, R, h.shape[-1]), emb.new_zeros(R, Lt, 1)
    terms = []
    for s in range(S):
        t = tok[:, s].contiguous()
        _, h, cell, _, cov, lv = dec.step(sent, h, cell, ea, ei, cov, mask_r, target=t)
        sent = emb_r[rows, t.clamp(0, Lt - 1)].unsqueeze(1)
        terms.append(lv)
    torch.stack(terms).sum().backward()


def run_workload(name, iters):
    from mmbidaf_b200 import ops
    from mmbidaf_b200.layers.encoding import length_plan
    from mmbidaf_b200.models import MMBiDAF
    from mmbidaf_b200.synth import make_batch
    c = WORKLOADS[name]
    dev = torch.device("cuda")
    torch.manual_seed(224)
    model = MMBiDAF(HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, dev, drop_prob=0.0, max_transcript_length=c["m"]).to(dev)
    b = make_batch(c["batch"], c["lt"], c["la"], c["li"], c["steps"], E_TEXT, E_AUDIO, E_IMAGE, seed=224).to(dev)
    S = c["steps"]
    res = {"workload": name, "shape": c, "arms": {}}
    dec = model.multimodal_att_decoder
    model.eval()
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    lens = length_plan(b.text_len, dev).len_i32.clone()
    key = ops.seed_key(224, dev)
    model.train()
    leaves = [t.detach().clone().requires_grad_() for t in (enc_a, enc_i, h0)]

    def timed(k, fn):
        for _ in range(3):
            fn()
        res["arms"][k] = stats(event_time(fn, iters))
        print(name, k, res["arms"][k]["median_ms"], flush=True)

    def forced_train(tokens):
        model.zero_grad(set_to_none=True)
        p_tok, terms = dec.force_train(b.text, leaves[2], leaves[0], leaves[1], mask, tokens)
        (p_tok.sum() + terms.sum()).backward()

    def by_hand(tokens):
        model.zero_grad(set_to_none=True)
        step_autograd(dec, b.text, leaves[2], leaves[0], leaves[1], mask, tokens)

    def by_hand_fused(tokens):
        saved = os.environ.get("MMB_DECODER_CUT")
        os.environ["MMB_DECODER_CUT"] = "fused"
        try:
            by_hand(tokens)
        finally:
            if saved is None:
                os.environ.pop("MMB_DECODER_CUT", None)
            else:
                os.environ["MMB_DECODER_CUT"] = saved

    def whole(tokens):
        model.zero_grad(set_to_none=True)
        sc = model.sequence_scores(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, S, tokens)
        (sc.logp.sum() + sc.loss.sum()).backward()

    for N in ARMS[name]:
        with torch.no_grad():
            _, tokens = dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, N, key)
        timed(f"N{N}_forced_train", lambda: forced_train(tokens))
        timed(f"N{N}_step_autograd", lambda: by_hand(tokens))
        timed(f"N{N}_step_autograd_fused", lambda: by_hand_fused(tokens))
        timed(f"N{N}_sequence_scores", lambda: whole(tokens))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_sequence_scores_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sequence_scores_bench: needs a CUDA device (no CPU timing)")
    import mmbidaf_b200
    mmbidaf_b200.set_precision(args.precision)
    out = {"gpu": gpu_info(), "precision": args.precision, "iters": args.iters, "workloads": []}
    for name in ([args.only] if args.only else list(WORKLOADS)):
        if name not in ARMS:
            continue
        out["workloads"].append(run_workload(name, args.iters))
        print(json.dumps(out["workloads"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
