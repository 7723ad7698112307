"""Summary scoring timings on one GPU: what the teacher-forced likelihood of N given candidates per video costs in one launch.

    python tools/score_bench.py [--out profiles/r09_score_bench.json] [--iters 20] [--precision fast|fp32]

Workloads as tools/summarize_bench.py (synthetic, seeded, four rotating batches of one padded-shape bucket):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 steps; N in 1, 4, 16
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 steps; N in 1, 4
On batch 0's encoder outputs, CUDA events, medians after a warm-up; the candidates are N sampled summaries per video:
  greedy_cluster     the greedy roll-out's cluster kernel (one launch, B clusters), the reference arm
  N{n}_sample        MultimodalAttentionDecoder.sample at the same N (one launch, B N clusters)
  N{n}_forced        MultimodalAttentionDecoder.force (one launch, B N clusters), p_tok and loss terms only
  N{n}_forced_probs  the same, also writing the (B, N, S, M) rows
  N4_host_loop       (cfg3) the same scores as a Python loop of the fused step kernel at B N rows, one launch per step
and at config-3 shapes the Summarizer.score replay per batch for N = 4 (CUDA events around the copies into the bucket and the replay).
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
from summarize_bench import E_AUDIO, E_IMAGE, E_TEXT, HIDDEN, N_ROTATE, WORKLOADS, event_time, gpu_info, stats  # noqa: E402

ARMS = {"cfg3": (1, 4, 16), "cfg5": (1, 4)}


def host_loop(dec, emb, h0, enc_a, enc_i, mask, tokens):
    """The forced roll-out as a Python loop: the fused step kernel over B N rows (the B-video tensors replicated) with each row's
    token as the target, then the gather of the next inputs."""
    from mmbidaf_b200 import ops
    B, N, S = tokens.shape
    rs = replicated(dec, enc_a, enc_i, N)
    Lt, H = rs.Lt, rs.H
    R = B * N
    tok = tokens.reshape(R, S)
    emb_r, mask_r = emb.repeat_interleave(N, 0), ops._u8(mask.bool().repeat_interleave(N, 0))
    rows = torch.arange(R, device=emb.device)
    sent, h = emb.new_zeros(R, emb.shape[2]), h0.reshape(B, H).repeat_interleave(N, 0).contiguous()
    cell, cov = torch.zeros(R, H, device=emb.device), torch.zeros(R, Lt, device=emb.device)
    for s in range(S):
        t = tok[:, s].contiguous()
        _, h, cell, _, cov, *_ = ops.decoder_step_fwd(rs, sent.contiguous(), h, cell, cov, mask_r, target=t)
        sent = emb_r[rows, t.clamp(0, Lt - 1)]


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
        if name == "cfg3":
            _, tok4 = dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, 4, key)
            with torch.no_grad():
                timed("N4_host_loop", lambda: host_loop(dec, b.text, h0, enc_a, enc_i, mask, tok4))
    finally:
        if saved is None:
            os.environ.pop("MMB_DECODER_CUT", None)
        else:
            os.environ["MMB_DECODER_CUT"] = saved
    for N in ARMS[name]:
        _, tokens = dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, N, key)
        timed(f"N{N}_sample", lambda: dec.sample(b.text, h0, enc_a, enc_i, mask, lens, S, N, key))
        timed(f"N{N}_forced", lambda: dec.force(b.text, h0, enc_a, enc_i, mask, tokens))
        timed(f"N{N}_forced_probs", lambda: dec.force(b.text, h0, enc_a, enc_i, mask, tokens, want_probs=True))
    if name == "cfg3":
        summarizer = Summarizer(model)
        cands = []
        for bb in batches:
            with torch.no_grad():
                ea, ei, hh, mm = model._encode(bb.text, bb.text_len, bb.audio, bb.audio_len, bb.images, bb.image_len, dec.prepare)
            cands.append(dec.sample(bb.text, hh, ea, ei, mm, length_plan(bb.text_len, dev).len_i32, S, 4, key)[1])
        for bb, tk in zip(batches, cands):
            summarizer.score(bb, tk)
        turn = iter(range(1 << 30))

        def replay():
            i = next(turn) % N_ROTATE
            summarizer.score(batches[i], cands[i])
        res["arms"]["N4_summarizer_score"] = stats(event_time(replay, iters))
        print(name, "N4_summarizer_score", res["arms"]["N4_summarizer_score"]["median_ms"], flush=True)
        model.eval()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_score_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_bench: needs a CUDA device (no CPU timing)")
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
