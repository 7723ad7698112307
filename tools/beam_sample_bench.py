"""Stochastic beam (samples without replacement) timings on one GPU: what ranking by Gumbel keys costs inside the beam roll-out.

    python tools/beam_sample_bench.py [--out profiles/r08_beam_sample_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/sample_bench.py (synthetic, seeded, four rotating batches of one padded-shape bucket):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 steps
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 steps
On batch 0's encoder outputs, CUDA events, medians of --iters after a warm-up:
  K{k}_stoch        MultimodalAttentionDecoder.beam_sample (one launch); cfg3: K in 1, 2, 4, 8; cfg5: K in 1, 2, 4
  K{k}_beam         MultimodalAttentionDecoder.beam at the same width, in the same run (the reference arm)
  K{k}_sample       MultimodalAttentionDecoder.sample with num_samples = K (with replacement), in the same run
  K4_stoch_constrained   K = 4 with no_repeat=True, min_sentences=3
  K4_host_loop      (cfg3) the same rule as a Python loop: the fused step kernel once per slot per step, the rule in torch ops
and at config-3 shapes the Summarizer replay + Summary.to_lists per batch for K = 4 (host clock, ends in the host copy).
Writes one JSON file with the GPU's name, power limit and max SM clock beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, N_ROTATE, WORKLOADS, event_time, gpu_info, host_time, stats  # noqa: E402

WIDTHS = {"cfg3": (1, 2, 4, 8), "cfg5": (1, 2, 4)}


def host_loop(dec, emb, h0, enc_a, enc_i, mask, S, K, key):
    """The unconstrained stochastic beam as a Python loop over the fused step kernel, with the normaliser, the keys and the ranking in
    torch ops on the device (the uniforms drawn by torch: the cost, not the bits, of the rule)."""
    from mmbidaf_b200 import ops
    seq = dec._sequence(enc_a, enc_i)["seq"]
    B, Lt, H, M = seq.B, seq.Lt, seq.H, seq.M
    dev = emb.device
    mask_u8 = ops._u8(mask)
    rows = torch.arange(B, device=dev)
    h = torch.zeros(B, K, H, device=dev)
    h[:, 0] = h0.reshape(B, H)
    cell, cov = torch.zeros(B, K, H, device=dev), torch.zeros(B, K, Lt, device=dev)
    tok = torch.zeros(B, K, dtype=torch.long, device=dev)
    phi, kk = torch.full((B, K), -math.inf, device=dev), torch.full((B, K), -math.inf, device=dev)
    phi[:, 0] = kk[:, 0] = 0
    for s in range(S):
        p = torch.zeros(B, K, M, device=dev)
        hn, cn, vn = torch.zeros_like(h), torch.zeros_like(cell), torch.zeros_like(cov)
        for k in range(K):
            sent = emb.new_zeros(B, emb.shape[2]) if s == 0 else emb[rows, tok[:, k].clamp(0, Lt - 1)]
            o = ops.decoder_step_fwd(seq, sent.contiguous(), h[:, k].contiguous(), cell[:, k].contiguous(), cov[:, k].contiguous(), mask_u8)
            p[:, k], hn[:, k], cn[:, k], vn[:, k] = o[0], o[1], o[2], o[4]
        cand = torch.isfinite(kk).unsqueeze(2) & (p > 0)
        l = torch.log(p)
        mu = torch.where(cand, l, -math.inf).max(2).values
        q = torch.where(cand, torch.floor(torch.exp(l - mu.unsqueeze(2)) * 16777216.0), 0.0)
        lam = mu + torch.log(q.sum(2) * 2.0 ** -24)
        G = phi.unsqueeze(2) + (l - lam.unsqueeze(2)) - torch.log(-torch.log(torch.rand(B, K, M, device=dev).clamp(2 ** -24, 1 - 2 ** -24)))
        Z = torch.where(cand, G, -math.inf).max(2).values
        a = G - Z.unsqueeze(2)
        v = (kk.unsqueeze(2) - G) + torch.where(a > -0.6931472, torch.log(-torch.expm1(a)), torch.log1p(-torch.exp(a)))
        ck = torch.where(cand, (kk.unsqueeze(2) - v.clamp_min(0)) - torch.log1p(torch.exp(-v.abs())), -math.inf)
        top = ck.reshape(B, -1).topk(K, 1)
        par = top.indices // M
        tok = top.indices % M
        kk = top.values
        phi = (phi.unsqueeze(2) + (l - lam.unsqueeze(2))).reshape(B, -1).gather(1, top.indices)
        g = par.view(B, K, 1)
        h, cell, cov = hn.gather(1, g.expand(B, K, H)), cn.gather(1, g.expand(B, K, H)), vn.gather(1, g.expand(B, K, Lt))


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

    for K in WIDTHS[name]:            # the three arms of a width side by side
        timed(f"K{K}_stoch", lambda: dec.beam_sample(b.text, h0, enc_a, enc_i, mask, lens, S, K, key))
        timed(f"K{K}_beam", lambda: dec.beam(b.text, h0, enc_a, enc_i, mask, lens, S, K))
        timed(f"K{K}_sample", lambda: dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, K, key))
    timed("K4_stoch_constrained", lambda: dec.beam_sample(b.text, h0, enc_a, enc_i, mask, lens, S, 4, key, 1.0, True, 3))
    if name == "cfg3":
        saved = os.environ.get("MMB_DECODER_CUT")
        os.environ["MMB_DECODER_CUT"] = "fused"
        try:
            with torch.no_grad():
                timed("K4_host_loop", lambda: host_loop(dec, b.text, h0, enc_a, enc_i, mask, S, 4, key))
        finally:
            if saved is None:
                os.environ.pop("MMB_DECODER_CUT", None)
            else:
                os.environ["MMB_DECODER_CUT"] = saved
        summarizer = Summarizer(model)
        fn = lambda bb: summarizer(bb, num_samples=4, replacement=False).to_lists()                 # noqa: E731
        for bb in batches:
            fn(bb)
        res["arms"]["K4_summarizer"] = stats(host_time(fn, batches, iters))
        print(name, "K4_summarizer", res["arms"]["K4_summarizer"]["median_ms"], flush=True)
        model.eval()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_beam_sample_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("beam_sample_bench: needs a CUDA device (no CPU timing)")
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
