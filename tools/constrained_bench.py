"""Constrained summarisation timings on one GPU: what repeat blocking and a minimum length cost inside the roll-out kernels.

    python tools/constrained_bench.py [--out profiles/constrained_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/summarize_bench.py (synthetic, seeded, four rotating batches of one padded-shape bucket):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 steps; beam widths 1, 2, 4, 8
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 steps; beam widths 1, 2, 4
Every arm runs twice: unconstrained, and with no_repeat=True, min_sentences=3 (suffix _constrained).  On batch 0's encoder outputs,
CUDA events, medians after a warm-up:
  greedy          MultimodalAttentionDecoder.greedy as summarize routes it: one launch of the cluster kernel, except at config 5
                  unconstrained, where B * Lt > 20 000 runs the chunk-parallel cut step by step (the constrained roll-out is always
                  the cluster kernel); greedy_cluster is the unconstrained cluster kernel forced, for a like-for-like comparison
  K{k}_beam       MultimodalAttentionDecoder.beam (one launch)
and at config-3 shapes the Summarizer replay + Summary.to_lists per batch (host clock, ends in the host copy) for greedy and K = 4.
Writes one JSON file with the GPU's name and power limit beside the numbers.
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

from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, N_ROTATE, WORKLOADS, event_time, gpu_info, host_time, stats  # noqa: E402

WIDTHS = {"cfg3": (1, 2, 4, 8), "cfg5": (1, 2, 4)}
CONSTRAINT = dict(no_repeat=True, min_sentences=3)
SETTINGS = (("", {}), ("_constrained", CONSTRAINT))


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
    res = {"workload": name, "shape": c, "rotating_batches": N_ROTATE, "constraint": CONSTRAINT,
           "greedy_unconstrained_cut": ops.decoder_cut(c["batch"], c["lt"]), "arms": {}}
    b = batches[0]
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    lens = length_plan(b.text_len, dev).len_i32.clone()

    def timed(key, fn):
        for _ in range(3):
            fn()
        res["arms"][key] = stats(event_time(fn, iters))
        print(name, key, res["arms"][key]["median_ms"], flush=True)

    for suffix, kw in SETTINGS:
        timed("greedy" + suffix, lambda: dec.greedy(b.text, h0, enc_a, enc_i, mask, S, text_len=lens, **kw))
    saved = os.environ.get("MMB_DECODER_CUT")
    os.environ["MMB_DECODER_CUT"] = "fused"
    try:
        timed("greedy_cluster", lambda: dec.greedy(b.text, h0, enc_a, enc_i, mask, S))
    finally:
        if saved is None:
            os.environ.pop("MMB_DECODER_CUT", None)
        else:
            os.environ["MMB_DECODER_CUT"] = saved
    for K in WIDTHS[name]:
        for suffix, kw in SETTINGS:
            timed(f"K{K}_beam{suffix}", lambda: dec.beam(b.text, h0, enc_a, enc_i, mask, lens, S, K, **kw))
    if name == "cfg3":
        for width in (None, 4):
            for suffix, kw in SETTINGS:
                summarizer = Summarizer(model)
                fn = lambda bb: summarizer(bb, beam_width=width, **kw).to_lists()                     # noqa: E731
                for bb in batches:
                    fn(bb)
                key = ("greedy" if width is None else f"K{width}") + "_summarizer" + suffix
                res["arms"][key] = stats(host_time(fn, batches, iters))
                print(name, key, res["arms"][key]["median_ms"], flush=True)
                model.eval()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "constrained_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("constrained_bench: needs a CUDA device (no CPU timing)")
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
