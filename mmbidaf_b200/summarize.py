"""Extractive summarisation (reference evaluate.py:107-126, :167-202, method='greedy') on the device.

``MMBiDAF.summarize`` runs the encoder half of the model, the whole greedy decode roll-out and the greedy sentence selection
without a host round trip; its result is a :class:`Summary`.  With ``beam_width=K`` the roll-out is a beam search over K
hypotheses per video (one launch too); the summary is the best hypothesis's, and :class:`Beams` holds all K.  With
``num_samples=N`` N summaries per video are drawn inside one launch (temperature, top-k, top-p); the summary is the likeliest sample's, and
:class:`Samples` holds all N.  ``no_repeat`` and ``min_sentences`` constrain any pick inside the roll-out kernel.
:class:`Summarizer` replays ``summarize`` from CUDA graphs, one capture per padded-shape bucket.  :func:`gather_summaries` collects the summaries of a data-parallel job on rank 0.
"""
from __future__ import annotations

import math
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from .ops import BEAM_MAX_WIDTH, check_sampling
from .synth import Batch

__all__ = ["Beams", "Inclusion", "Samples", "Summary", "Summarizer", "gather_summaries"]


def check_options(who: str, with_targets: bool, beam_width, no_repeat, min_sentences, num_samples=None, temperature=1.0, top_k=0,
                  seed=None, top_p=1.0, replacement=True) -> None:
    """The decode options of ``MMBiDAF.summarize`` / ``Summarizer``, checked before any device work: ``beam_width`` None or an int
    in 1..8, ``no_repeat`` a bool, ``min_sentences`` an int >= 0; neither a beam nor a constraint with targets (the eval loss is
    defined by the unconstrained greedy roll-out).  Sampling: ``num_samples`` None or an int in 1..64, not with a beam or targets;
    ``temperature`` finite and > 0, ``top_k`` an int in 0..8, ``seed`` None or an int, ``top_p`` a real in (0, 1] -- set only with
    ``num_samples``.  ``replacement`` a bool; False (the stochastic beam) needs ``num_samples`` in 1..8 and takes neither ``top_k``
    nor ``top_p``."""
    if not isinstance(replacement, bool):
        raise ValueError(f"{who}: replacement {replacement!r}, expected a bool")
    if not replacement:
        if num_samples is None:
            raise ValueError(f"{who}: replacement=False without num_samples")
        if isinstance(num_samples, bool) or not isinstance(num_samples, int) or not 1 <= num_samples <= BEAM_MAX_WIDTH:
            raise ValueError(f"{who}: num_samples {num_samples!r} with replacement=False, expected an int in 1..{BEAM_MAX_WIDTH}")
        if isinstance(top_k, bool) or top_k != 0 or isinstance(top_p, bool) or top_p != 1.0:
            raise ValueError(f"{who}: top_k / top_p with replacement=False -- the stochastic beam draws from every candidate")
    if num_samples is not None:
        check_sampling(who, num_samples, temperature, top_k, top_p)
        if beam_width is not None:
            raise ValueError(f"{who}: num_samples with beam_width -- sampling and beam search are separate decodes")
        if with_targets:
            raise ValueError(f"{who}: num_samples with targets -- the eval loss is defined by the greedy roll-out")
        if seed is not None and (isinstance(seed, bool) or not isinstance(seed, int)):
            raise ValueError(f"{who}: seed {seed!r}, expected None or an int")
    elif temperature != 1.0 or top_k != 0 or seed is not None or isinstance(top_p, bool) or top_p != 1.0:
        raise ValueError(f"{who}: temperature / top_k / top_p / seed without num_samples")
    if beam_width is not None:
        if isinstance(beam_width, bool) or not isinstance(beam_width, int) or not 1 <= beam_width <= BEAM_MAX_WIDTH:
            raise ValueError(f"{who}: beam_width {beam_width!r}, expected None or an int in 1..{BEAM_MAX_WIDTH}")
        if with_targets:
            raise ValueError(f"{who}: beam_width with targets -- the eval loss is defined by the greedy roll-out")
    if not isinstance(no_repeat, bool):
        raise ValueError(f"{who}: no_repeat {no_repeat!r}, expected a bool")
    if isinstance(min_sentences, bool) or not isinstance(min_sentences, int) or min_sentences < 0:
        raise ValueError(f"{who}: min_sentences {min_sentences!r}, expected an int >= 0")
    if with_targets and (no_repeat or min_sentences > 0):
        raise ValueError(f"{who}: no_repeat / min_sentences with targets -- the eval loss is defined by the unconstrained roll-out")


def _select(tokens: Sequence[int], text_len: int) -> List[int]:
    """The greedy_search rule (decode.greedy_search, evaluate.py:185-202) over a token row: the EOS row text_len - 1 ends the
    summary, an index past it is skipped, any other is kept."""
    chosen = []
    for k in tokens:
        if k == text_len - 1:
            break
        if k > text_len - 1:
            continue
        chosen.append(int(k))
    return chosen


class Beams(NamedTuple):
    """Every slot of a beam roll-out (``MMBiDAF.summarize(..., beam_width=K)``, the rule at mmb_decoder_beam_fused in
    include/mmbidaf_b200.h).  Slot j of step s holds the j-th best hypothesis after that step."""
    tokens: torch.Tensor                   # (B, S, K) int64: the slot's last token (-1: empty slot)
    parents: torch.Tensor                  # (B, S, K) int32: the slot of step s - 1 it extends (-1: empty slot)
    scores: torch.Tensor                   # (B, S, K) fp32: the sum of logf(p) along its path (-inf: empty slot)
    probs: torch.Tensor                    # (B, S, K, M) fp32: the distribution its parent produced at step s (zero for carries / empty)

    def paths(self) -> List[List[Tuple[List[int], float]]]:
        """Per video, the token rows of the non-empty slots after the last step, best first, with their scores (host lists)."""
        tok, par, sc = self.tokens.cpu(), self.parents.cpu(), self.scores.cpu()
        B, S, K = tok.shape
        out = []
        for b in range(B):
            hyps = []
            for j in range(K):
                if int(par[b, S - 1, j]) < 0:
                    continue
                row, k = [], j
                for s in range(S - 1, -1, -1):
                    row.append(int(tok[b, s, k]))
                    k = int(par[b, s, k])
                hyps.append((row[::-1], float(sc[b, S - 1, j])))
            out.append(hyps)
        return out

    def n_best(self, text_len: Sequence[int]) -> List[List[Tuple[List[int], float]]]:
        """Per video, the hypotheses of the last step's non-empty slots, best first: (chosen sentence indices under the greedy_search
        rule, score).  ``text_len`` (B) gives each video's EOS row (text_len - 1)."""
        lens = [int(n) for n in (text_len.tolist() if torch.is_tensor(text_len) else text_len)]
        return [[(_select(row, lens[b]), score) for row, score in hyps] for b, hyps in enumerate(self.paths())]


class Samples(NamedTuple):
    """Every sampled roll-out (``MMBiDAF.summarize(..., num_samples=N)``, the rule at mmb_decoder_sample_fused in
    include/mmbidaf_b200.h)."""
    tokens: torch.Tensor                   # (B, N, S) int64: the picks of sample n of video b
    probs: torch.Tensor                    # (B, N, S, M) fp32: its distribution at every step
    logp: torch.Tensor                     # (B, N) fp32: sum of log p_s[tok_s] up to and including its first EOS pick (all S without)

    def summaries(self, text_len: Sequence[int]) -> List[List[Tuple[List[int], float]]]:
        """Per video, every sample in order: (chosen sentence indices under the greedy_search rule, logp).  ``text_len`` (B) gives
        each video's EOS row (text_len - 1)."""
        lens = [int(n) for n in (text_len.tolist() if torch.is_tensor(text_len) else text_len)]
        tok, lp = self.tokens.cpu().tolist(), self.logp.cpu().tolist()
        return [[(_select(row, lens[b]), lp[b][n]) for n, row in enumerate(rows)] for b, rows in enumerate(tok)]


def sample_logp(probs: torch.Tensor, tokens: torch.Tensor, text_len_i32: torch.Tensor) -> torch.Tensor:
    """logp (B, N) fp32 of sampled roll-outs: the sum of log p_s[tok_s] over the steps up to and including the first EOS pick
    (text_len - 1), or over all S without one.  Device ops only (capturable)."""
    lp = torch.log(probs.gather(3, tokens.clamp_min(0).unsqueeze(3)).squeeze(3))               # (B, N, S)
    hit = (tokens == (text_len_i32.long() - 1).view(-1, 1, 1)).long()
    after = (hit.cumsum(2) - hit) > 0                                                          # steps after the first EOS pick
    return torch.where(after, torch.zeros_like(lp), lp).sum(2)


def best_sample(samples: Samples, sel: torch.Tensor, count: torch.Tensor):
    """The likeliest sample of every video (highest logp, ties to the lower n): (its distributions (B, S, M), its indices (B, S) and
    count (B) out of ``sel`` (B N, S) / ``count`` (B N), the greedy selection over every sample's tokens)."""
    B, N, S = samples.tokens.shape
    best = samples.logp.argmax(1)                          # the first maximal n
    rows = torch.arange(B, device=best.device)
    return samples.probs[rows, best], sel.view(B, N, S)[rows, best], count.view(B, N)[rows, best]


class Inclusion(NamedTuple):
    """What a sample without replacement (``MMBiDAF.summarize(..., num_samples=K, replacement=False)``, the rule at
    mmb_decoder_beam_sample_fused in include/mmbidaf_b200.h) needs for estimates under the model: per final slot its log-probability
    under the sampling distribution and its key, and per video the threshold.  Empty slots have logq = keys = -inf."""
    logq: torch.Tensor                     # (B, K) fp32: phi of every final slot, the log-probability of its sequence
    keys: torch.Tensor                     # (B, K) fp32: its perturbed log-probability (descending over the slots)
    threshold: torch.Tensor                # (B) fp32: kappa, the (K + 1)-th key of all sequences (-inf when at most K exist)

    def probabilities(self) -> torch.Tensor:
        """(B, K) fp64: the probability that each sample is in a sample of K, 1 - exp(-exp(logq - threshold)); 1 where the threshold
        is -inf (every sequence is in), 0 for empty slots.  Device ops only (capturable)."""
        lq, th = self.logq.double(), self.threshold.double().unsqueeze(1)
        p = -torch.expm1(-torch.exp(lq - th))
        p = torch.where(th == -math.inf, torch.ones_like(p), p)
        return torch.where(lq == -math.inf, torch.zeros_like(p), p)

    def weights(self, normalise: bool = True) -> torch.Tensor:
        """(B, K) fp64 importance weights exp(logq) / probabilities() (0 for empty slots): sum_i w_i f(y_i) is an unbiased estimate
        of the expectation of f under the sampling distribution; ``normalise`` divides each video's weights by their sum (a
        consistent estimate with lower variance).  Device ops only (capturable)."""
        q = self.probabilities()
        w = torch.where(q > 0, torch.exp(self.logq.double()) / q, torch.zeros_like(q))
        return w / w.sum(1, keepdim=True) if normalise else w


class Summary(NamedTuple):
    out_distributions: torch.Tensor        # (B, S, M) fp32: every step's distribution over the sentences, as MMBiDAF.forward returns
    loss: Optional[torch.Tensor]           # the eval loss (models.py:197-199) when targets were given, else None
    indices: torch.Tensor                  # (B, S) int32: the chosen sentence indices of every video, padded with -1
    counts: torch.Tensor                   # (B) int32: how many of them are valid
    beams: Optional[Beams] = None          # a beam summary's every slot (then out_distributions are the best path's rows), else None
    samples: Optional[Samples] = None      # a sampled summary's every sample (then the other fields are the likeliest sample's), else None
    inclusion: Optional[Inclusion] = None  # a sample without replacement's inclusion probabilities and weights, else None

    def to_lists(self) -> List[List[int]]:
        """The chosen sentence indices per video as host lists (copies only ``indices`` and ``counts``):
        equal to ``decode.get_generated_indices(out_distributions, text_len)``."""
        idx, cnt = self.indices.cpu(), self.counts.cpu().tolist()
        return [idx[b, :c].tolist() for b, c in enumerate(cnt)]


def _bucket_key(batch: Batch, with_targets: bool, beam_width: Optional[int], no_repeat: bool = False, min_sentences: int = 0,
                sampling: tuple = (None, 1.0, 0, None, 1.0, True)):
    return (tuple(batch.text.shape), tuple(batch.audio.shape), tuple(batch.images.shape), int(batch.max_dec_len),
            tuple(batch.targets.shape) if with_targets else None, beam_width, no_repeat, min_sentences, sampling)


class _Bucket:
    """One captured ``summarize``: static inputs, static length plans, the graph and its (static) result."""

    def __init__(self, model, batch: Batch, with_targets: bool, warmup: int, beam_width: Optional[int] = None,
                 no_repeat: bool = False, min_sentences: int = 0, sampling: tuple = (None, 1.0, 0, None, 1.0, True)):
        import gc
        from .layers.encoding import pin_lengths
        dev = batch.text.device
        # private copies: the captured kernels read the inputs and the lengths from these fixed addresses
        self.batch = Batch(batch.text.clone(), list(batch.text_len), batch.audio.clone(), list(batch.audio_len), batch.images.clone(),
                           list(batch.image_len), batch.targets.clone(), list(batch.target_len), batch.max_dec_len)
        self.with_targets = with_targets
        self.beam_width = beam_width
        self.no_repeat, self.min_sentences = no_repeat, min_sentences
        self.sampling = sampling             # (num_samples, temperature, top_k, seed, top_p, replacement); seed None: the key state exists after warm-up
        self.plans = [pin_lengths(lst, dev) for lst in (self.batch.text_len, self.batch.audio_len, self.batch.image_len)]
        for m in model.modules():          # per-sequence caches of eager calls still own tensors (see Trainer.capture)
            if hasattr(m, "_cache"):
                m._cache = None
        gc.collect()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):        # module loads, per-shape constants (decode_loss weights), the plans' masks
                self._run(model)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.result = self._run(model)

    def _run(self, model) -> Summary:
        for plan in self.plans:            # inside the captured region: lengths -> int32, order, masks
            plan.refresh()
        b = self.batch
        return model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, b.max_dec_len,
                               b.targets if self.with_targets else None, beam_width=self.beam_width, no_repeat=self.no_repeat,
                               min_sentences=self.min_sentences, num_samples=self.sampling[0], temperature=self.sampling[1],
                               top_k=self.sampling[2], seed=self.sampling[3], top_p=self.sampling[4], replacement=self.sampling[5])

    def load(self, batch: Batch) -> None:
        if batch is self.batch:
            return
        for plan, lens in zip(self.plans, (batch.text_len, batch.audio_len, batch.image_len)):
            plan.update(lens)
        s = self.batch
        s.text.copy_(batch.text, non_blocking=True)
        s.audio.copy_(batch.audio, non_blocking=True)
        s.images.copy_(batch.images, non_blocking=True)
        if self.with_targets:
            s.targets.copy_(batch.targets, non_blocking=True)


class Summarizer:
    """``model.summarize`` replayed from CUDA graphs.  A batch of a padded-shape bucket seen before (text, audio and key-frame widths,
    the batch size, ``max_dec_len``, with targets their width, the beam width and the constraints) is copied into that bucket's static inputs, its
    lengths into the bucket's static length plans, and the bucket's graph is replayed; a new bucket is captured first (after ``warmup`` eager runs).
    The decoder's weight layouts are rebuilt inside the graph, so in-place parameter updates (an optimiser step) show up on the next
    replay.  The returned :class:`Summary` holds the bucket's static output tensors: the next replay of the same bucket overwrites them."""

    def __init__(self, model, warmup: int = 2):
        self.model = model
        self.warmup = warmup
        self.buckets: Dict[tuple, _Bucket] = {}

    def __call__(self, batch: Batch, with_targets: bool = False, beam_width: Optional[int] = None, no_repeat: bool = False,
                 min_sentences: int = 0, num_samples: Optional[int] = None, temperature: float = 1.0, top_k: int = 0,
                 seed: Optional[int] = None, top_p: float = 1.0, replacement: bool = True) -> Summary:
        """``batch`` resident on the device; ``with_targets`` also computes the eval loss from ``batch.targets``; ``beam_width``
        decodes by beam search, ``no_repeat`` / ``min_sentences`` constrain the pick (``MMBiDAF.summarize``); each width and each
        setting of the constraints in its own bucket.  ``num_samples`` / ``temperature`` / ``top_k`` / ``seed`` / ``top_p`` sample (each setting,
        the seed included, in its own bucket): with ``seed=None`` every replay draws a fresh key from the device key stream, with an int
        seed every replay gives that seed's samples.  ``replacement=False`` samples without replacement (the stochastic beam, its own
        buckets).  The options are checked before anything is copied or captured."""
        check_options("Summarizer", with_targets, beam_width, no_repeat, min_sentences, num_samples, temperature, top_k, seed, top_p,
                      replacement)
        sampling = (num_samples, temperature, top_k, seed, top_p, replacement)
        key = _bucket_key(batch, with_targets, beam_width, no_repeat, min_sentences, sampling)
        bucket = self.buckets.get(key)
        if bucket is None:
            bucket = self.buckets[key] = _Bucket(self.model, batch, with_targets, self.warmup, beam_width, no_repeat, min_sentences,
                                                 sampling)
        else:
            bucket.load(batch)
        bucket.graph.replay()
        return bucket.result


def gather_summaries(summary: Summary, group=None) -> Optional[List[List[int]]]:
    """The summaries of a data-parallel job on rank 0: every rank holds the summary of its contiguous shard of the batch
    (``trainer.shard_batch``, which keeps the global text padding -- the decoder's attention runs over every padded text position,
    quirk Q2, so a narrower shard would change the picks).  Rank 0 gets the chosen indices of every video in batch order, as
    ``Summary.to_lists`` of the whole batch would give them; the other ranks get None.  One all-gather of the shard sizes, then one
    all-gather of the (count, indices) rows padded to the largest shard, as int32 tensors on the summary's device."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return summary.to_lists()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    idx, cnt = summary.indices, summary.counts
    B, S = idx.shape
    size = torch.tensor([B], dtype=torch.int32, device=idx.device)
    sizes = [torch.empty_like(size) for _ in range(world)]
    dist.all_gather(sizes, size, group=group)
    sizes = [int(t) for t in sizes]
    rows = torch.full((max(sizes), S + 1), -1, dtype=torch.int32, device=idx.device)
    rows[:B, 0] = cnt
    rows[:B, 1:] = idx
    parts = [torch.empty_like(rows) for _ in range(world)]
    dist.all_gather(parts, rows, group=group)
    if rank != 0:
        return None
    out = []
    for n, part in zip(sizes, parts):
        host = part[:n].cpu()
        out += [host[b, 1:1 + int(host[b, 0])].tolist() for b in range(n)]
    return out
