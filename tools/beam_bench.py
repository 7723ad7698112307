"""Beam-search summarisation timings on one GPU: what K hypotheses per video cost against the greedy roll-out.

    python tools/beam_bench.py [--out profiles/beam_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/summarize_bench.py (synthetic, seeded, four rotating batches of one padded-shape bucket):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 steps; widths 1, 2, 4, 8
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 steps; widths 1, 2, 4
Arms per width:
  beam_kernel     the beam roll-out alone (MultimodalAttentionDecoder.beam: one launch), CUDA events, on batch 0's encoder outputs
  host_loop       the same roll-out as a host loop: the fused step kernel once per slot and step, log / sort / gathers in between
                  (tests/test_beam_gpu.py's reference), CUDA events
  summarizer      Summarizer replay with beam_width=K + Summary.to_lists, host clock per batch (ends in the host copy)
and once per workload greedy_kernel: the greedy roll-out (one launch of the cluster kernel), CUDA events.  Every width's tables are
compared with the host loop's, bit for bit.  Writes one JSON file with the GPU's name and power limit beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, N_ROTATE, WORKLOADS, event_time, gpu_info, host_time, stats  # noqa: E402

WIDTHS = {"cfg3": (1, 2, 4, 8), "cfg5": (1, 2, 4)}


def run_workload(name, iters):
    from mmbidaf_b200.layers.encoding import length_plan
    from mmbidaf_b200.models import MMBiDAF
    from mmbidaf_b200.summarize import Summarizer
    from mmbidaf_b200.synth import make_batch
    from test_beam_gpu import _reference
    c = WORKLOADS[name]
    dev = torch.device("cuda")
    torch.manual_seed(224)
    model = MMBiDAF(HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, dev, drop_prob=0.2, max_transcript_length=c["m"]).to(dev)
    model.eval()
    batches = [make_batch(c["batch"], c["lt"], c["la"], c["li"], c["steps"], E_TEXT, E_AUDIO, E_IMAGE, seed=224 + i).to(dev)
               for i in range(N_ROTATE)]
    S = c["steps"]
    res = {"workload": name, "shape": c, "rotating_batches": N_ROTATE, "arms": {}, "beam_equal_to_host_loop": {}}
    b = batches[0]
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    lens = length_plan(b.text_len, dev).len_i32.clone()
    saved = os.environ.get("MMB_DECODER_CUT")
    os.environ["MMB_DECODER_CUT"] = "fused"             # the greedy kernel and the host loop's step kernel: the cluster cut, as the beam
    try:
        greedy = lambda: dec.greedy(b.text, h0, enc_a, enc_i, mask, S)     # noqa: E731
        for _ in range(3):
            greedy()
        res["arms"]["greedy_kernel"] = stats(event_time(greedy, iters))
        for K in WIDTHS[name]:
            beam = lambda: dec.beam(b.text, h0, enc_a, enc_i, mask, lens, S, K)                       # noqa: E731
            loop = lambda: _reference(dec, b.text, h0, enc_a, enc_i, mask, lens, S, K)                 # noqa: E731
            for _ in range(2):
                got, want = beam(), loop()
            res["beam_equal_to_host_loop"][f"K{K}"] = all(torch.equal(g, w) for g, w in zip(got[:4], want))
            res["arms"][f"K{K}_beam_kernel"] = stats(event_time(beam, iters))
            res["arms"][f"K{K}_host_loop"] = stats(event_time(loop, max(3, iters // 4)))
            print(name, K, res["arms"][f"K{K}_beam_kernel"]["median_ms"], res["arms"][f"K{K}_host_loop"]["median_ms"], flush=True)
    finally:
        if saved is None:
            os.environ.pop("MMB_DECODER_CUT", None)
        else:
            os.environ["MMB_DECODER_CUT"] = saved
    for K in WIDTHS[name]:
        summarizer = Summarizer(model)
        fn = lambda bb: summarizer(bb, beam_width=K).to_lists()                                       # noqa: E731
        for bb in batches:
            fn(bb)
        res["arms"][f"K{K}_summarizer"] = stats(host_time(fn, batches, iters))
        model.eval()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "beam_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("beam_bench: needs a CUDA device (no CPU timing)")
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
