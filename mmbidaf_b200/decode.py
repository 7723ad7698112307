"""Extractive decoding over the model's output distributions (reference evaluate.py:167-202)."""
from __future__ import annotations

from typing import List, Sequence

import numpy as np
import torch


def greedy_search(out_distributions: torch.Tensor, original_text_length: int) -> List[int]:
    """Sentence indices picked for one video: arg-max per timestep until it hits the EOS row
    ``original_text_length - 1`` (evaluate.py:185-202).  The reference looks every pick up in the transcript on disk
    (``get_source_sentence``, :236-259): an index past the transcript yields no sentence and is skipped, not a stop
    (:195, :255-256) -- reproduced here from the length alone (the transcript has ``original_text_length - 1`` sentences)."""
    picks = out_distributions.argmax(dim=1).tolist()
    chosen = []
    for k in picks:
        if k == original_text_length - 1:
            break
        if k > original_text_length - 1:
            continue
        chosen.append(int(k))
    return chosen


def nucleus(p, eligible=None, top_k: int = 0, top_p: float = 1.0) -> List[int]:
    """The candidates a sampled pick draws from (the rules at mmb_decoder_sample_fused / mmb_decoder_sample_nucleus_fused in
    include/mmbidaf_b200.h), in (p descending, m ascending) order, from one row ``p`` (M) of fp32 probabilities as the kernels write
    them: every m (or those with ``eligible[m]`` set), cut to the first ``top_k`` when ``top_k > 0``, then for ``top_p < 1`` to the
    first n whose integer masses q = floor(p 2^24) reach P Q (P = rint(top_p 2^24) in fp32, Q the candidates' mass), n >= 1.
    Integers only after the fp32 inputs, so the set is the kernels' exactly.  A verification helper (O(M log M) on the host, one row
    at a time): the tests check the kernels' picks against it, and a user can check a returned sample the same way."""
    row = np.asarray(p.detach().cpu() if torch.is_tensor(p) else p, dtype=np.float32).reshape(-1)
    ok = np.ones(row.shape, dtype=bool) if eligible is None else np.asarray(
        eligible.detach().cpu() if torch.is_tensor(eligible) else eligible, dtype=bool).reshape(-1)
    cand = sorted((m for m in range(row.size) if ok[m]), key=lambda m: (-float(row[m]), m))
    if top_k > 0:
        cand = cand[:top_k]
    if np.float32(top_p) == np.float32(1.0):
        return cand
    q = [int(np.floor(np.float64(row[m]) * 2 ** 24)) for m in cand]     # exact: p 2^24 is a scaled fp32 value
    P = int(np.rint(np.float64(np.float32(top_p)) * 2 ** 24))           # half to even, as rintf
    need, acc = P * sum(q), 0
    for n, qm in enumerate(q, 1):
        acc += qm
        if (acc << 24) >= need:
            return cand[:n]
    return cand                                                          # (no candidate)


def truncated_key(parent_key, g, z):
    """The child key of the stochastic beam rule (mmb_decoder_beam_sample_fused in include/mmbidaf_b200.h) in numpy fp32: the
    perturbed log-probability ``g`` of a child truncated to at most its parent's key ``parent_key``, given ``z``, the largest ``g`` of
    the parent's children -- key' = (parent_key - max(v, 0)) - log1p(exp(-|v|)), v = (parent_key - g) + log1mexp(g - z),
    log1mexp(a) = log(-expm1(a)) above -ln 2, else log1p(-exp(a)).  The child with g = z keeps parent_key exactly; the result is
    monotone in g.  ``g`` may be an array.  (numpy's log1p / expm1 may round differently from the device's in the last bit.)"""
    f = np.float32
    kp, gv, zv = f(parent_key), np.asarray(g, dtype=f), f(z)
    a = gv - zv
    with np.errstate(divide="ignore", invalid="ignore"):
        l1 = np.where(a > f(-0.6931472), np.log(-np.expm1(a)), np.log1p(-np.exp(a))).astype(f)
        v = (kp - gv) + l1
        return ((kp - np.maximum(v, f(0))) - np.log1p(np.exp(-np.abs(v)))).astype(f)


def get_generated_indices(batch_out_distributions: torch.Tensor, original_text_lengths: Sequence[int]) -> List[List[int]]:
    """Greedy indices for a batch (B, T, M) (evaluate.py:167-183, method='greedy')."""
    host = batch_out_distributions.detach().cpu()
    return [greedy_search(host[b], int(original_text_lengths[b])) for b in range(host.shape[0])]
