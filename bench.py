#!/usr/bin/env python
"""bench.py -- MMBiDAF training throughput on B200 (BASELINE.json metric) + fused-BiDAF roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W]                # our arm (N>1: launched by torchrun)
    python bench.py --impl reference [--steps K] [--warmup W]          # the reference's own code on the host CPU
    python bench.py --dump-outputs DIR                                 # also write the last timed step's results as DIR/<name>.npy

One "step" = one pass of the hot path over one batch of synthetic Coursera-shaped videos:
forward -> loss.backward() -> gradient all-reduce(SUM) -> clip_grad_norm_(2.0) -> Adadelta(lr 0.5).step()
(reference train.py:146-155) on BASELINE config 3 (B=32 videos per GPU, Lt<=409, La<=1024, Li<=128,
T_dec<=12, hidden 100, text 300 / audio 128 / image 1000, drop 0.2).  At N GPUs every rank runs the same
per-GPU batch (weak scaling; N=8 is BASELINE config 4's global batch of 256); `cfg4_strong` in the same line is
config 4 as stated: a global batch of 256 sharded 256/N per GPU.

One JSON line on stdout (rank 0).
  value        videos/s, inputs resident in HBM, the step replayed from CUDA graphs over FOUR rotating batches with different
               length draws (the collator pads every batch to its own maxima and lengths change every batch, datasets.py:298-302)
  e2e          the same step fed from pinned host memory (H2D inside the timed region), every step's loss copied to the host and read
               there (one step late, under the next step; the last one inside the timed region)
  no_graph     the same step launched kernel by kernel from Python (no CUDA graph)
  fp32_tier    the rel <= 1e-5 tier (fp32 FFMA BiDAF kernels, fp32 library GEMMs)
  roofline     the fused BiDAF forward on BASELINE config 2 (B=64, Lc=512, Lq=256, d=200), CUDA events in this run, against
               the measured HBM peak; its backward beside it
  cfg5         long-lecture evaluate.py-style decoding (B=16, Lt=La=4096, Li=2048, 16 greedy steps, no_grad)
  eager_cuda   the UNMODIFIED reference (oracle/_ref, staged by oracle/stage_ref.py) in torch eager on the same B200
  cpu_baseline the unmodified reference on this box's host cores (bounded sample)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, M = 100, 300, 128, 1000, 409
CFG3 = dict(batch=32, lt=409, la=1024, li=128, t_dec=12)            # per GPU
CFG2 = dict(batch=64, lc=512, lq=256, d=200)
CFG4_GLOBAL = 256
CFG5 = dict(batch=16, lt=4096, la=4096, li=2048, m=4096, steps=16)
DROP = 0.2                                                           # train.py:209
METRIC, UNIT = "mmbidaf_train_videos_per_s", "videos/s"
N_ROTATE = 4
DUMP_LIMIT = 64 << 20                                                # bytes --dump-outputs may write


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid = torch.cuda.get_device_properties(index).uuid
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as exc:                                           # pragma: no cover
            self.nv, self.error = None, repr(exc)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "sw_power_cap": 0x4}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.reasons.update(k for k, v in names.items() if bits & v)
            except Exception:
                pass
            time.sleep(0.004)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def workload_config(n_gpus: int, **over):
    cfg = {"workload": "BASELINE config 3: full MMBiDAF training step (embedding->RNNEncoder->BiDAFx2->mod-LSTM->"
                       "multimodal attention decoder->loss; backward; clip 2.0; Adadelta lr 0.5)",
           "per_gpu_batch": CFG3["batch"], "global_batch": CFG3["batch"] * n_gpus, "max_text_len": CFG3["lt"],
           "max_audio_len": CFG3["la"], "max_image_len": CFG3["li"], "max_dec_len": CFG3["t_dec"], "hidden": HIDDEN,
           "embed": [E_TEXT, E_AUDIO, E_IMAGE], "max_transcript_length": M, "drop_prob": DROP,
           "parallelism": f"dp{n_gpus}",
           "launch": f"step captured once into CUDA graphs (one padded-shape bucket) and replayed over {N_ROTATE} rotating batches "
                     "with different length draws",
           "l2": "inputs+activations per step exceed L2 (126 MB); BiDAF microbench rotates 4 input sets (4 x 144 MB)"}
    cfg.update(over)
    return cfg


def dump_outputs(directory: str, arrays: dict) -> None:
    """Write every tensor of ``arrays`` as ``directory/<name>.npy`` in float32 (float64 stays float64).  The inputs of a run are
    seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the limit of {DUMP_LIMIT}")
    os.makedirs(directory, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------
# The reference itself (oracle/_ref: the unmodified models.py + layers/, staged by oracle/stage_ref.py) -- on the host CPU
# (--impl reference, cpu_baseline) and in torch eager on the GPU (eager_cuda).  If the staged copy is missing the CPU legs
# fall back to the oracle's functional port (kind "port").  The only place besides tests/ and smoke() that executes oracle/.
# ------------------------------------------------------------------------------------------------------
def _reference_step_fn(device, batch_size: int, drop: float):
    from mmbidaf_b200.synth import make_batch
    from oracle import ref_loader
    torch.manual_seed(224)
    model = ref_loader.build_model("reference", HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, device, drop, M)
    model.train()
    opt = torch.optim.Adadelta(model.parameters(), lr=0.5)                      # train.py:110
    batches = [make_batch(batch_size, CFG3["lt"], CFG3["la"], CFG3["li"], CFG3["t_dec"], E_TEXT, E_AUDIO, E_IMAGE,
                          seed=224 + i).to(device) for i in range(N_ROTATE)]
    state = {"k": 0}

    def step():
        b = batches[state["k"] % N_ROTATE]
        state["k"] += 1
        opt.zero_grad()
        _, loss = model(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, b.targets, b.target_len, b.max_dec_len)
        loss.backward()                                                         # train.py:148
        torch.nn.utils.clip_grad_norm_(model.parameters(), 2.0)                 # train.py:154
        opt.step()
        return loss
    return step


def cpu_training_throughput(videos_per_step: int, steps: int, warmup: int):
    """-> (videos/s, ms/step, cores, kind, sample description)."""
    from oracle import ref_loader
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    shapes = (f"{videos_per_step} videos/step of config 3 shapes (Lt<=409, La<=1024, Li<=128, T_dec<=12), {N_ROTATE} rotating batches, "
              f"{steps} timed + {warmup} warm-up steps, fwd+bwd+clip+Adadelta, fp32, dropout {DROP}, torch CPU {torch.__version__}")
    if ref_loader.available():
        step = _reference_step_fn(torch.device("cpu"), videos_per_step, DROP)
        kind, what = "reference", "the unmodified reference (oracle/_ref/models.py + layers/, nn.LSTM on PackedSequence): "
    else:                                                                       # staged copy missing: the functional port
        from mmbidaf_b200.synth import make_batch
        from oracle import mmbidaf_oracle as O
        params = {k: v.clone().requires_grad_(True) for k, v in O.make_params(HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, M).items()}
        plist = list(params.values())
        opt = torch.optim.Adadelta(plist, lr=0.5)
        batch = make_batch(videos_per_step, CFG3["lt"], CFG3["la"], CFG3["li"], CFG3["t_dec"], E_TEXT, E_AUDIO, E_IMAGE, seed=224)
        img = batch.images.flatten(2)

        def step():
            opt.zero_grad()
            _, loss = O.mmbidaf_forward(params, batch.text, batch.text_len, batch.audio, batch.audio_len, img, batch.image_len,
                                        batch.targets, batch.max_dec_len, M, training=True, fast_lstm=True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(plist, 2.0)
            opt.step()
        kind, what = "port", "oracle port (oracle/_ref not staged; dropout off): "
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    total = time.perf_counter() - t0
    return videos_per_step * steps / total, total / steps * 1e3, cores, kind, what + shapes


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vps, ms, cores, kind, sample = cpu_training_throughput(CFG3["batch"], args.steps, max(args.warmup, 1))
    line = {"impl": "reference", "metric": METRIC, "value": round(vps, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": round(ms, 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, parallelism="host CPU, one process", global_batch=CFG3["batch"],
                                      launch="torch eager on the host CPU (the reference's own code path), all host threads",
                                      l2="n/a (CPU)"),
            "cpu_baseline": {"value": round(vps, 4), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(vps, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def _event_time(fn, iters: int) -> float:
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3 / iters


def _cfg2_sets(device, gen):
    B, Lc, Lq, d = CFG2["batch"], CFG2["lc"], CFG2["lq"], CFG2["d"]
    sets = []
    for _ in range(4):                                      # 4 x 144 MB > L2: every timed forward reads cold data
        c = torch.randn(B, Lc, d, generator=gen).to(device)
        q = torch.randn(B, Lq, d, generator=gen).to(device)
        c_len = torch.randint(Lc // 2, Lc + 1, (B,), generator=gen)
        q_len = torch.randint(Lq // 2, Lq + 1, (B,), generator=gen)
        cm = (torch.arange(Lc).unsqueeze(0) < c_len.unsqueeze(1)).to(device)
        qm = (torch.arange(Lq).unsqueeze(0) < q_len.unsqueeze(1)).to(device)
        sets.append((c, q, cm, qm))
    return sets


def bidaf_microbench(device, rounds: int, warmup: int, precision: int, backward: bool = False):
    """Fused BiDAF forward (or backward) on BASELINE config 2; returns (avg seconds per call, algorithmic bytes).
    The four calls over the four rotating input sets are captured into ONE CUDA graph and the graph is replayed: at ~50 us per
    call the Python / ctypes overhead of launching from the host (~40 us) would otherwise be part of the measurement."""
    from mmbidaf_b200 import ops
    B, Lc, Lq, d = CFG2["batch"], CFG2["lc"], CFG2["lq"], CFG2["d"]
    gen = torch.Generator().manual_seed(224)
    sets = _cfg2_sets(device, gen)
    w = [torch.randn(d, generator=gen).to(device) * 0.1 for _ in range(3)]
    bias = torch.zeros(1, device=device)
    if backward:                                             # saved forward state + an upstream gradient per input set
        full = []
        for s in sets:
            out, q2c, lse_r, lse_c, bm, ws = ops.bidaf_fwd(s[0], s[1], s[2], s[3], w[0], w[1], w[2], bias,
                                                            precision=precision, save=True)
            full.append(s + (torch.randn(out.shape, generator=gen).to(device), out, q2c, lse_r, lse_c, bm, ws))
        sets = full
        run = lambda s: ops.bidaf_bwd(s[4], s[0], s[1], s[2], s[3], w[0], w[1], w[2], bias, None, None, 1.0, s[5], s[9], s[6], s[7],
                                      s[8], s[10], precision)
    else:
        # aux=False: the forward as the layer runs it under no_grad (only `out`; T and the log-sum-exps are saved for a backward pass only)
        run = lambda s: ops.bidaf_fwd(s[0], s[1], s[2], s[3], w[0], w[1], w[2], bias, precision=precision, aux=False)
    side = torch.cuda.Stream(device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(max(warmup, 3)):
            run(sets[i % 4])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        keep = [run(s) for s in sets]                        # outputs stay alive in the graph's pool
    for _ in range(3):
        graph.replay()
    seconds = _event_time(graph.replay, rounds) / 4
    del keep
    algo_bytes = 4 * B * (Lc * d + Lq * d + Lc * 4 * d) + B * (Lc + Lq)            # SURVEY.md 8d
    if backward:                                            # read dX (4 Lc d), c, q; write dc, dq
        algo_bytes = 4 * B * (4 * Lc * d + 2 * Lc * d + 2 * Lq * d)
    return seconds, algo_bytes


def lstm_microbench(device, rounds: int = 5):
    """One bidirectional LSTM layer of the metric's longest recurrence (audio_enc of config 3: B=32, L=1024, in=H=100) through the
    layer op (input GEMM + persistent recurrence kernel; backward: BPTT kernel + weight-gradient GEMMs), captured into a CUDA graph.
    SURVEY 8d: the recurrence is serial-latency bound -- reported as us per time step next to its (low) share of the HBM roofline.
    Algorithmic bytes per layer (SURVEY 8d): activations 4 B L (in + 2H) + weights 2 * 4 (4H in + 4H H + 8H); forward + backward = 2 x."""
    from mmbidaf_b200 import functional as Fn
    B, L, H = CFG3["batch"], CFG3["la"], HIDDEN
    gen = torch.Generator().manual_seed(11)
    lengths = torch.randint(L // 2, L + 1, (B,), generator=gen)
    lengths[0] = L
    len_d = lengths.to(torch.int32).to(device)
    ord_d = torch.argsort(lengths, descending=True).to(torch.int32).to(device)
    ws = [((torch.rand(*shape, generator=gen) - 0.5) * 0.2).to(device).requires_grad_(True) for _ in range(2)
          for shape in ((4 * H, H), (4 * H, H), (4 * H,), (4 * H,))]
    x = torch.randn(B, L, H, generator=gen).to(device).requires_grad_(True)
    g_out = torch.randn(B, L, 2 * H, generator=gen).to(device)

    def fwd():
        with torch.no_grad():
            return Fn.lstm_layer(x, len_d, ord_d, ws)[0]

    def fwd_bwd():
        out, _ = Fn.lstm_layer(x, len_d, ord_d, ws)
        return torch.autograd.grad(out, [x] + ws, g_out)

    res = {}
    for name, fn in (("fwd", fwd), ("fwd_bwd", fwd_bwd)):
        side = torch.cuda.Stream(device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            keep = fn()
        graph.replay()
        res[name] = _event_time(graph.replay, rounds)
        del keep, graph
    algo = 4 * B * L * (H + 2 * H) + 2 * 4 * (4 * H * H + 4 * H * H + 8 * H)
    return res["fwd"], res["fwd_bwd"], algo, (B, L, H)


def measured_traffic(name: str):
    """DRAM bytes per launch of the roofline kernel from the committed ncu capture of this round (profiles/*.json written by
    tools/ncu_traffic.py from `ncu --set full`), or None: never a literal in this file."""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None
    with open(path) as f:
        blob = json.load(f)
    return int(blob["dram_bytes_read"] + blob["dram_bytes_write"])


def cfg5_timing(device):
    """BASELINE config 5: long-lecture stress, evaluate.py:107-126 flow (eval mode, no_grad, 16 greedy steps)."""
    from mmbidaf_b200.models import MMBiDAF
    from mmbidaf_b200.synth import make_batch
    c = CFG5
    torch.manual_seed(224)
    model = MMBiDAF(HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, device, drop_prob=DROP, max_transcript_length=c["m"]).to(device)
    model.eval()
    batch = make_batch(c["batch"], c["lt"], c["la"], c["li"], c["steps"], E_TEXT, E_AUDIO, E_IMAGE, seed=224).to(device)

    def run():
        with torch.no_grad():
            return model(batch.text, batch.text_len, batch.audio, batch.audio_len, batch.images, batch.image_len, batch.targets,
                         batch.target_len, c["steps"])
    for _ in range(2):
        run()
    seconds = _event_time(run, 3)
    d = 2 * HIDDEN
    bidaf_bytes = sum(4 * c["batch"] * (c["lt"] * d + lq * d + c["lt"] * 4 * d) + c["batch"] * (c["lt"] + lq)
                      for lq in (c["la"], c["li"]))
    return {"workload": "BASELINE config 5: B=16, Lt=La=4096, Li=2048, M=4096, eval, 16 greedy steps, no_grad",
            "ms": round(seconds * 1e3, 2), "videos_per_s": round(c["batch"] / seconds, 1),
            "bidaf_algorithmic_bytes": bidaf_bytes}


def eager_cuda_baselines(device):
    """The unmodified reference modules (oracle/_ref) in torch eager on this GPU (cuBLAS + cuDNN + ATen): the library bar of
    SURVEY.md section 2.2 -- the full config-3 training step and the BiDAF op at config 2.  PyTorch's default precision flags
    (fp32 matmul, TF32 allowed inside cuDNN)."""
    from oracle import ref_loader
    if not ref_loader.available():
        return {"unavailable": "oracle/_ref is not staged"}
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, True
    try:
        step = _reference_step_fn(device, CFG3["batch"], DROP)
        for _ in range(2):
            step()
        t_step = _event_time(step, 4)
        _, ref_att, _ = ref_loader.load("reference")
        gen = torch.Generator().manual_seed(224)
        sets = _cfg2_sets(device, gen)
        mod = ref_att.BiDAFAttention(CFG2["d"], drop_prob=DROP).to(device)
        mod.eval()
        k = {"i": 0}

        def fwd():
            s = sets[k["i"] % 4]
            k["i"] += 1
            with torch.no_grad():
                return mod(*s)
        for _ in range(3):
            fwd()
        t_fwd = _event_time(fwd, 12)
        mod.train()
        grads = [torch.randn(CFG2["batch"], CFG2["lc"], 4 * CFG2["d"], device=device)]
        leaves = [(s[0].clone().requires_grad_(True), s[1].clone().requires_grad_(True), s[2], s[3]) for s in sets]

        def fwd_bwd():
            s = leaves[k["i"] % 4]
            k["i"] += 1
            out = mod(*s)
            torch.autograd.grad(out, (s[0], s[1], *mod.parameters()), grads[0])
        for _ in range(3):
            fwd_bwd()
        t_fb = _event_time(fwd_bwd, 8)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved
    return {"what": "the unmodified reference (oracle/_ref) in torch eager on the same GPU, fp32 matmul / cuDNN LSTM",
            "step_videos_per_s": round(CFG3["batch"] / t_step, 2), "step_ms": round(t_step * 1e3, 2),
            "bidaf_cfg2_fwd_us": round(t_fwd * 1e6, 1), "bidaf_cfg2_fwd_bwd_us": round(t_fb * 1e6, 1), "torch": torch.__version__}


def run_gpu_arm(args):
    import torch.distributed as dist
    import mmbidaf_b200
    from mmbidaf_b200 import ops
    from mmbidaf_b200.models import MMBiDAF
    from mmbidaf_b200.synth import Batch, make_batch
    from mmbidaf_b200.trainer import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout (NCCL_DEBUG=VERSION in this image): keep stdout to the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    mmbidaf_b200.set_precision(args.precision)
    sections = set(args.sections.split(","))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        start.record()
        for _ in range(steps):
            fn()
        end.record()
        barrier()
        ms = torch.tensor([start.elapsed_time(end)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)        # max over ranks
        return float(ms.item()) / 1e3

    def new_trainer(seed=224):
        torch.manual_seed(seed)                              # args.py:43-46
        model = MMBiDAF(HIDDEN, E_TEXT, E_AUDIO, E_IMAGE, device, drop_prob=DROP, max_transcript_length=M).to(device)
        return Trainer(model)

    def batches_of(per_gpu):
        hosts = [make_batch(per_gpu, CFG3["lt"], CFG3["la"], CFG3["li"], CFG3["t_dec"], E_TEXT, E_AUDIO, E_IMAGE,
                            seed=224 + 101 * rank + i).pin() for i in range(N_ROTATE)]
        return hosts, [h.to(device) for h in hosts]

    work = torch.cuda.Stream(device)                         # never the legacy stream: the step is graph-captured
    torch.cuda.set_stream(work)
    trainer = new_trainer()
    hosts, residents = batches_of(CFG3["batch"])
    assert len({(tuple(h.text_len), tuple(h.audio_len)) for h in hosts}) == N_ROTATE      # different length draws ...
    assert all(h.text.shape == hosts[0].text.shape and h.max_dec_len == hosts[0].max_dec_len for h in hosts)   # ... one bucket
    launches0 = ops.launch_count
    for i in range(args.warmup):
        trainer.step(residents[i % N_ROTATE])
    launches_per_step = (ops.launch_count - launches0) // max(args.warmup, 1)
    graphed = not args.no_graph
    turn = {"k": 0}
    if graphed:
        # the step is ~1200 launches (launch-bound): forward + backward + gradient pack are captured once, clip + Adadelta once
        # (the NCCL all-reduce sits between the two graphs); every replay takes the NEXT batch: its tensors are copied into the
        # graph's static inputs and its lengths into the static length plans (layers/encoding.py::LengthPlan)
        trainer.capture(residents[0], warmup=1)

    def run_resident():
        b = residents[turn["k"] % N_ROTATE]
        turn["k"] += 1
        turn["loss"] = trainer.step_graphed(b) if graphed else trainer.step(b)

    for _ in range(N_ROTATE):
        run_resident()
    with ClockSampler(local) as clocks:
        seconds = timed(run_resident, args.steps)
    if args.dump_outputs and rank == 0:
        # what a caller of the step holds after the last timed step (the sections below keep training the same model)
        arrays = {"loss": turn["loss"], "grad_norm": trainer.last_grad_norm}
        for name, p in trainer.model.named_parameters():
            arrays["param." + name] = p
            arrays["grad." + name] = p.grad
        dump_outputs(args.dump_outputs, arrays)
    launches = launches_per_step * args.steps
    videos = CFG3["batch"] * world * args.steps

    # kernel-by-kernel launch from Python of the same step (no CUDA graph), same rotating batches
    no_graph = None
    if graphed and "step" in sections:
        def run_eager():
            b = residents[turn["k"] % N_ROTATE]
            turn["k"] += 1
            return trainer.step(b)
        run_eager()
        n_eager = max(3, min(args.steps, 8))
        t = timed(run_eager, n_eager)
        no_graph = {"value": round(CFG3["batch"] * world * n_eager / t, 2), "unit": UNIT, "ms_per_step": round(t / n_eager * 1e3, 3),
                    "steps": n_eager}

    # End-to-end: every step's inputs start in pinned host memory and its loss is read back by the host.  The copy
    # of step k+1 is issued on a side stream while step k computes (a two-slot device staging area), the way an
    # input pipeline would feed the model; all of it happens inside the timed region.
    copy_stream = torch.cuda.Stream(device)
    slots = [hosts[0].to(device), hosts[0].to(device)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"k": 0}

    def prefetch(k):
        slot, host = slots[k & 1], hosts[k % N_ROTATE]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k & 1])                       # the step that last read this slot is done
            for dst, src in ((slot.text, host.text), (slot.audio, host.audio), (slot.images, host.images),
                             (slot.targets, host.targets)):
                dst.copy_(src, non_blocking=True)                        # H2D from pinned memory
            ready[k & 1].record(copy_stream)

    # The loss of every step is copied to pinned host memory and read by the host -- one step late: the copy of step k is awaited after
    # step k + 1 has been enqueued, so the host never idles the GPU between two graph replays waiting for four bytes.  The last step's
    # loss is read inside the timed region too (`flush`).
    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event(), torch.cuda.Event()]
    pending = {"k": None, "seen": []}

    def read_pending():
        if pending["k"] is not None:
            j = pending["k"] & 1
            loss_ready[j].synchronize()
            pending["seen"].append(float(loss_host[j][0]))               # the host reads the step's loss
            pending["k"] = None

    def e2e_step(last=False):
        k = state["k"]
        slot, host = slots[k & 1], hosts[k % N_ROTATE]
        torch.cuda.current_stream().wait_event(ready[k & 1])
        feed = Batch(slot.text, host.text_len, slot.audio, host.audio_len, slot.images, host.image_len, slot.targets,
                     host.target_len, host.max_dec_len)
        loss = trainer.step_graphed(feed) if graphed else trainer.step(feed)
        consumed[k & 1].record()
        loss_host[k & 1].copy_(loss.detach().reshape(1), non_blocking=True)      # D2H read of the step's loss
        loss_ready[k & 1].record()
        prefetch(k + 1)
        state["k"] = k + 1
        read_pending()                                                   # step k - 1's loss, while step k runs
        pending["k"] = k
        if last:
            read_pending()

    e2e_seconds = float("nan")
    if "e2e" in sections:
        for ev in consumed:
            ev.record()
        prefetch(0)
        for _ in range(max(2, args.warmup // 2)):
            e2e_step()
        read_pending()
        calls = {"n": 0}

        def e2e_timed():
            calls["n"] += 1
            e2e_step(last=calls["n"] == args.steps)
        e2e_seconds = timed(e2e_timed, args.steps)
        assert len(pending["seen"]) >= args.steps and all(v == v for v in pending["seen"])    # every step's loss reached the host

    # BASELINE config 4 as stated: a global batch of 256 videos sharded over the ranks (strong scaling)
    cfg4 = None
    per_gpu4 = CFG4_GLOBAL // world
    if "cfg4" in sections and graphed and per_gpu4 * world == CFG4_GLOBAL:
        if per_gpu4 == CFG3["batch"]:
            cfg4 = {"global_batch": CFG4_GLOBAL, "per_gpu_batch": per_gpu4, "value": round(videos / seconds, 2), "unit": UNIT,
                    "ms_per_step": round(seconds / args.steps * 1e3, 3), "note": "identical to the main measurement at this N"}
        else:
            tr4 = new_trainer()
            _, res4 = batches_of(per_gpu4)
            for i in range(2):
                tr4.step(res4[i])
            tr4.capture(res4[0], warmup=1)
            k4 = {"k": 0}

            def run4():
                k4["k"] += 1
                return tr4.step_graphed(res4[k4["k"] % N_ROTATE])
            for _ in range(2):
                run4()
            n4 = max(3, min(args.steps, 6))
            t4 = timed(run4, n4)
            cfg4 = {"global_batch": CFG4_GLOBAL, "per_gpu_batch": per_gpu4, "value": round(CFG4_GLOBAL * n4 / t4, 2), "unit": UNIT,
                    "ms_per_step": round(t4 / n4 * 1e3, 3), "steps": n4, "scaling": "strong"}
            del tr4, res4

    line = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        fast = args.precision == "fast"
        prec = ops.PREC_BF16 if fast else ops.PREC_FP32
        line = {"metric": METRIC, "value": round(videos / seconds, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(seconds / args.steps * 1e3, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16 tcgen05 BiDAF + tf32 library GEMMs, fp32 accumulate / soft-max / LSTM" if fast else "f32",
                "data": "synthetic", "config": workload_config(world), "clocks": clocks.summary(),
                "e2e": {"value": round(videos / e2e_seconds, 2), "unit": UNIT, "h2d_bytes_per_step": hosts[0].h2d_bytes(),
                        "d2h_bytes_per_step": 4, "ms_per_step": round(e2e_seconds / args.steps * 1e3, 3)},
                "gpu_launches": launches}
        if not graphed:
            line["config"]["launch"] = "every kernel launched from Python (--no-graph)"
        if no_graph is not None:
            line["no_graph"] = no_graph
        if cfg4 is not None:
            line["cfg4_strong"] = cfg4
        if "bidaf" in sections:
            t_bidaf, algo = bidaf_microbench(device, 10, 5, prec)
            achieved = algo / t_bidaf / 1e9
            roof = {"kernel": ("fused BiDAF forward, tcgen05 bf16 tier (bidaf_pack_kernel + the main tcgen05 launch)" if fast
                               else "fused BiDAF forward, fp32 tier (bidaf_pass_f32 x2)")
                              + ", BASELINE config 2 (B=64, Lc=512, Lq=256, d=200)",
                    "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                    "traffic": measured_traffic("r02_bidaf_fwd_traffic.json") if fast else None,
                    "peak_source": peak_src, "algorithmic_bytes": algo, "us_per_forward": round(t_bidaf * 1e6, 1),
                    "timing": "CUDA events around replays of one CUDA graph holding the 4 calls over 4 rotating input sets"}
            if fast:
                t_bwd, algo_bwd = bidaf_microbench(device, 10, 5, ops.PREC_BF16, backward=True)
                roof["backward"] = {"us": round(t_bwd * 1e6, 1), "algorithmic_bytes": algo_bwd,
                                    "achieved": round(algo_bwd / t_bwd / 1e9, 1), "frac": round(algo_bwd / t_bwd / 1e9 / peak, 4),
                                    "traffic": measured_traffic("r02_bidaf_bwd_traffic.json")}
                fb = (algo + algo_bwd) / (t_bidaf + t_bwd) / 1e9
                roof["forward_backward"] = {"us": round((t_bidaf + t_bwd) * 1e6, 1), "algorithmic_bytes": algo + algo_bwd,
                                            "achieved": round(fb, 1), "frac": round(fb / peak, 4)}
            t_lf, t_lfb, algo_l, (lb, ll, lh) = lstm_microbench(device)
            roof["lstm"] = {"kernel": f"one bidirectional LSTM layer (input GEMM + bilstm_fwd_kernel; backward: bilstm_bwd_kernel + weight-"
                                      f"gradient GEMMs), audio_enc of config 3: B={lb}, L={ll}, in=H={lh}",
                            "bound": "serial latency (SURVEY 8d): one dependent (4H x H) mat-vec + gate non-linearities per time step",
                            "fwd_us": round(t_lf * 1e6, 1), "fwd_us_per_timestep": round(t_lf * 1e6 / ll, 3),
                            "fwd_bwd_us": round(t_lfb * 1e6, 1), "fwd_bwd_us_per_timestep": round(t_lfb * 1e6 / ll, 3),
                            "algorithmic_bytes_fwd": algo_l, "hbm_frac_fwd": round(algo_l / t_lf / 1e9 / peak, 4),
                            "hbm_frac_fwd_bwd": round(2 * algo_l / t_lfb / 1e9 / peak, 4)}
            line["roofline"] = roof
        if "cfg5" in sections:
            line["cfg5"] = cfg5_timing(device)
        if "fp32" in sections and fast and graphed and world == 1:
            mmbidaf_b200.set_precision("fp32")
            try:
                tr32 = new_trainer()
                for i in range(2):
                    tr32.step(residents[i])
                tr32.capture(residents[0], warmup=1)
                k32 = {"k": 0}

                def run32():
                    k32["k"] += 1
                    return tr32.step_graphed(residents[k32["k"] % N_ROTATE])
                for _ in range(2):
                    run32()
                n32 = max(3, min(args.steps, 6))
                t32 = _event_time(run32, n32)
                line["fp32_tier"] = {"value": round(CFG3["batch"] / t32, 2), "unit": UNIT, "ms_per_step": round(t32 * 1e3, 3),
                                     "dtype": "f32 (FFMA BiDAF kernels, fp32 library GEMMs): rel <= 1e-5 tier", "steps": n32}
                del tr32
            finally:
                mmbidaf_b200.set_precision(args.precision)
        if world == 1 and "eager" in sections:
            try:
                line["eager_cuda"] = eager_cuda_baselines(device)
            except Exception as exc:                                     # the bar must not take the bench line down with it
                line["eager_cuda"] = {"unavailable": repr(exc)[:200]}
        if world == 1 and not args.no_cpu_baseline:
            # bounded sample: a reference CPU step at the full batch of 32 takes ~8 s, so 1 warm-up + 3 timed steps (~30 s)
            vps, _, cores, kind, sample = cpu_training_throughput(CFG3["batch"], 3, 1)
            line["cpu_baseline"] = {"value": round(vps, 4), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--precision", default="fast", choices=["fast", "fp32"],
                    help="fast: bf16 tensor-core BiDAF + TF32 GEMMs (rel<=2e-2); fp32: rel<=1e-5 tier")
    ap.add_argument("--sections", default="step,e2e,cfg4,bidaf,cfg5,fp32,eager", help="profiling aid: which GPU sections to run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss, gradient norm, parameters and gradients as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
