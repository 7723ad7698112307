"""Summarisation timings on one GPU (evaluate.py:107-126, :167-202, greedy): what a batch of extractive summaries costs.

    python tools/summarize_bench.py [--out profiles/summarize_bench.json] [--iters 20] [--precision fast|fp32] [--only cfg3|cfg5]

Two workloads, each with four rotating batches of one padded-shape bucket (synthetic, seeded):
  cfg3  config-3 shapes in eval: B=32, Lt 409, La 1024, Li 128, M 409, 12 greedy steps
  cfg5  config 5: B=16, Lt=La=4096, Li=2048, M=4096, 16 greedy steps
Arms, each per batch and ending with the chosen sentence indices on the host (a host clock around work that ends in a device
synchronise, after warm-up runs of every batch):
  a  forward   eval() + no_grad MMBiDAF.forward, then decode.get_generated_indices (copies the (B, S, M) distributions)
  b  eager     MMBiDAF.summarize + Summary.to_lists
  c  graph     Summarizer replay + Summary.to_lists
  d  the decoder roll-out alone on the same encoder outputs, CUDA events: the greedy cluster kernel (one launch), the per-step loop
     of forward (step kernel + arg-max + gather per step) and, at cfg5, the chunk-parallel cut step by step
The picks of every arm are compared with arm a's.  Writes one JSON file with the GPU's name and power limit beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HIDDEN, E_TEXT, E_AUDIO, E_IMAGE = 100, 300, 128, 1000
WORKLOADS = {
    "cfg3": dict(batch=32, lt=409, la=1024, li=128, m=409, steps=12),
    "cfg5": dict(batch=16, lt=4096, la=4096, li=2048, m=4096, steps=16),
}
N_ROTATE = 4


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def host_time(fn, batches, iters):
    """Seconds per batch: host clock around `iters` rounds over the rotating batches, each ending in a host copy (a synchronise)."""
    times = []
    for i in range(iters):
        b = batches[i % len(batches)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(b)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return times


def event_time(fn, iters):
    times = []
    for _ in range(iters):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        fn()
        end.record()
        end.synchronize()
        times.append(start.elapsed_time(end) / 1e3)
    return times


def stats(times):
    ms = [t * 1e3 for t in times]
    return {"mean_ms": round(statistics.mean(ms), 3), "median_ms": round(statistics.median(ms), 3), "min_ms": round(min(ms), 3),
            "max_ms": round(max(ms), 3), "n": len(ms)}


def run_workload(name, iters):
    from mmbidaf_b200.decode import get_generated_indices
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

    def arm_a(b):
        with torch.no_grad():
            out, _ = model(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, b.targets, b.target_len, S)
        return get_generated_indices(out, b.text_len)

    def arm_b(b):
        return model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, S).to_lists()

    summarizer = Summarizer(model)

    def arm_c(b):
        return summarizer(b).to_lists()

    res = {"workload": name, "shape": c, "rotating_batches": N_ROTATE, "decoder_cut": None, "arms": {}}
    picks = {}
    for arm, fn in (("a_forward_get_generated_indices", arm_a), ("b_summarize_eager", arm_b), ("c_summarizer_graph", arm_c)):
        picks[arm] = [fn(b) for b in batches]          # warm-up of every batch (and the capture of arm c)
        res["arms"][arm] = stats(host_time(fn, batches, iters))
        model.eval()
    ref = picks["a_forward_get_generated_indices"]
    res["picks_equal_arm_a"] = {arm: p == ref for arm, p in picks.items()}

    # d: the roll-out alone, on the encoder outputs of batch 0
    from mmbidaf_b200 import ops
    b = batches[0]
    dec = model.multimodal_att_decoder
    B, Lt = b.text.shape[:2]
    res["decoder_cut"] = ops.decoder_cut(B, Lt)
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
        rows = torch.arange(B, device=dev)

        def step_loop():                                  # what forward's eval loop launches (models.py:254-266)
            h, cell = h0, h0.new_zeros(1, B, HIDDEN)
            cov, inp = h0.new_zeros(B, Lt, 1), b.text.new_zeros(B, 1, E_TEXT)
            outs = []
            for _ in range(S):
                p, h, cell, _, cov, _ = dec.step(inp, h, cell, enc_a, enc_i, cov, mask)
                inp = b.text[rows, p.max(dim=1)[1]].unsqueeze(1)
                outs.append(p)
            return torch.stack(outs).transpose(0, 1)

        saved = os.environ.get("MMB_DECODER_CUT")
        arms_d = {"greedy_kernel": ("fused", lambda: dec.greedy(b.text, h0, enc_a, enc_i, mask, S)[0]),
                  "step_loop_fused_step": ("fused", step_loop)}
        if name == "cfg5":
            arms_d["greedy_chunk_cut"] = ("chunks", lambda: dec.greedy(b.text, h0, enc_a, enc_i, mask, S)[0])
            arms_d["step_loop_chunk_cut"] = ("chunks", step_loop)
        outs = {}
        try:
            for arm, (cut, fn) in arms_d.items():
                os.environ["MMB_DECODER_CUT"] = cut
                for _ in range(3):
                    outs[arm] = fn()
                res["arms"]["d_rollout_" + arm] = stats(event_time(fn, iters))
        finally:
            if saved is None:
                os.environ.pop("MMB_DECODER_CUT", None)
            else:
                os.environ["MMB_DECODER_CUT"] = saved
        # (bit for bit: the greedy kernel against the loop of step kernels; the chunk cut against its own loop)
        res["rollout_equal_to_step_loop"] = {"greedy_kernel": bool(torch.equal(outs["greedy_kernel"], outs["step_loop_fused_step"]))}
        if "greedy_chunk_cut" in outs:
            res["rollout_equal_to_step_loop"]["greedy_chunk_cut"] = bool(torch.equal(outs["greedy_chunk_cut"], outs["step_loop_chunk_cut"]))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "summarize_bench.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"])
    ap.add_argument("--only", choices=sorted(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("summarize_bench: needs a CUDA device (no CPU timing)")
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
