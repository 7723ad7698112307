"""Sampled summarisation timings on one GPU: what N drawn roll-outs per video cost inside one launch.

    python tools/sample_bench.py [--out profiles/r06_sample_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/summarize_bench.py (synthetic, seeded, four rotating batches of one padded-shape bucket):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 steps; N in 1, 4, 16, top_k in 0, 8
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 steps; N in 1, 4, top_k 0
On batch 0's encoder outputs, CUDA events, medians after a warm-up:
  greedy_cluster   the greedy roll-out's cluster kernel (one launch), the reference arm
  greedy_x4        the same kernel over the B videos replicated four times (B 4 videos): what N = 4 samples would cost as greedy
  N{n}_k{k}        MultimodalAttentionDecoder.sample (one launch); _constrained with no_repeat=True, min_sentences=3
  N4_host_loop     (cfg3) the same 4 samples as a Python loop of the fused step kernel at B N rows and mmb_sample_pick per step
and at config-3 shapes the Summarizer replay + Summary.to_lists per batch for N = 4 (host clock, ends in the host copy).
Writes one JSON file with the GPU's name, power limit and max SM clock beside the numbers.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, N_ROTATE, WORKLOADS, event_time, gpu_info, host_time, stats  # noqa: E402

ARMS = {"cfg3": ((1, 0), (4, 0), (16, 0), (1, 8), (4, 8), (16, 8)), "cfg5": ((1, 0), (4, 0))}


def replicated(dec, enc_a, enc_i, N):
    """The decoder's per-sequence tensors of the B videos, each row repeated N times (B N rows)."""
    from mmbidaf_b200 import _lib
    seq = dec._sequence(enc_a, enc_i)["seq"]
    rs = copy.copy(seq)
    for f in ("proj_a", "proj_i", "enc_a", "enc_i"):
        setattr(rs, f, getattr(seq, f).repeat_interleave(N, 0).contiguous())
    rs.B, rs.nch = seq.B * N, _lib.lib().mmb_decoder_chunks(seq.B * N, seq.Lt)
    rs.counters = torch.zeros(2, seq.B * N, device=enc_a.device, dtype=torch.int32)
    return rs


def host_loop(dec, emb, h0, enc_a, enc_i, mask, S, N, key):
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
        sent = emb_r[rows, ops.sample_pick(p, key, base, S, s, N).clamp(0, Lt - 1)]


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

    saved = os.environ.get("MMB_DECODER_CUT")
    os.environ["MMB_DECODER_CUT"] = "fused"
    try:
        timed("greedy_cluster", lambda: dec.greedy(b.text, h0, enc_a, enc_i, mask, S))
        with torch.no_grad():
            rs = replicated(dec, enc_a, enc_i, 4)
            emb4, h4 = b.text.repeat_interleave(4, 0).contiguous(), h0.reshape(h0.shape[0], -1).repeat_interleave(4, 0).contiguous()
            mask4 = ops._u8(mask.bool().repeat_interleave(4, 0))
            timed("greedy_x4", lambda: ops.decoder_greedy_fwd(rs, emb4, h4, mask4, S))
        if name == "cfg3":
            with torch.no_grad():
                timed("N4_host_loop", lambda: host_loop(dec, b.text, h0, enc_a, enc_i, mask, S, 4, key))
    finally:
        if saved is None:
            os.environ.pop("MMB_DECODER_CUT", None)
        else:
            os.environ["MMB_DECODER_CUT"] = saved
    for N, top_k in ARMS[name]:
        timed(f"N{N}_k{top_k}", lambda: dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, N, key, 1.0, top_k))
    for top_k in ((0, 8) if name == "cfg3" else (0,)):
        timed(f"N4_k{top_k}_constrained", lambda: dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, 4, key, 1.0, top_k, True, 3))
    if name == "cfg3":
        summarizer = Summarizer(model)
        fn = lambda bb: summarizer(bb, num_samples=4).to_lists()                                    # noqa: E731
        for bb in batches:
            fn(bb)
        res["arms"]["N4_summarizer"] = stats(host_time(fn, batches, iters))
        print(name, "N4_summarizer", res["arms"]["N4_summarizer"]["median_ms"], flush=True)
        model.eval()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_sample_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench: needs a CUDA device (no CPU timing)")
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
