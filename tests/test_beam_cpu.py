"""CPU: the host side of beam summaries -- Beams.paths / Beams.n_best (backtracking and the greedy_search rule) on hand-built tables,
and Summary's optional beams field."""
import math

import torch

from mmbidaf_b200.decode import greedy_search
from mmbidaf_b200.summarize import Beams, Summary

NEG = -math.inf


def _beams(tokens, parents, scores, M=6):
    t = torch.tensor(tokens, dtype=torch.int64)
    return Beams(t, torch.tensor(parents, dtype=torch.int32), torch.tensor(scores, dtype=torch.float32),
                 torch.zeros(*t.shape, M))


def test_backtrack_follows_the_parents():
    # one video, S = 3, K = 2; slot 0 of the last step descends from slot 1 of step 1, which descends from slot 0 of step 0
    b = _beams([[[2, 3], [4, 1], [0, 5]]],
               [[[0, 0], [1, 0], [1, 0]]],
               [[[-0.1, -0.5], [-0.6, -0.7], [-0.8, -0.9]]])
    assert b.paths() == [[([2, 1, 0], _f32(-0.8)), ([3, 4, 5], _f32(-0.9))]]
    # EOS row 5 (text_len 6): the second hypothesis stops at it
    assert b.n_best([6]) == [[([2, 1, 0], _f32(-0.8)), ([3, 4], _f32(-0.9))]]


def _f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


def test_carries_after_eos_and_empty_slots():
    # K = 3, S = 3, EOS row 1 (text_len 2): two candidates at step 0 only, so slot 2 stays empty; slot 0 picks EOS at step 0 and is
    # carried (token 1, parent 0) after it
    b = _beams([[[1, 0, -1], [1, 0, -1], [1, 0, -1]]],
               [[[0, 0, -1], [0, 1, -1], [0, 1, -1]]],
               [[[-0.2, -1.8, NEG], [-0.2, -2.5, NEG], [-0.2, -3.0, NEG]]])
    hyps = b.n_best([2])[0]
    assert len(hyps) == 2                                  # the empty slot is no hypothesis
    assert hyps[0] == ([], _f32(-0.2))                     # the best path finishes at step 0: an empty summary
    assert hyps[1] == ([0, 0, 0], _f32(-3.0))


def test_ties_keep_the_slot_order_and_each_video_its_own_eos():
    # two videos, equal scores in both slots: the order of the slots is the order of the list
    b = _beams([[[3, 2], [3, 2]], [[0, 4], [1, 1]]],
               [[[0, 0], [1, 0]], [[0, 0], [0, 1]]],
               [[[-1.0, -1.0], [-2.0, -2.0]], [[-0.5, -0.5], [-0.5, -0.5]]])
    nb = b.n_best(torch.tensor([5, 2], dtype=torch.int32))
    assert nb[0] == [([2, 3], -2.0), ([3, 2], -2.0)]
    # video 1, EOS row 1: slot 0 = [0, 1] -> [0]; slot 1 = [4, 1]: 4 lies past the transcript and is skipped -> []
    assert nb[1] == [([0], -0.5), ([], -0.5)]


def test_n_best_applies_the_greedy_search_rule():
    g = torch.Generator().manual_seed(3)
    S, K, M = 7, 3, 9
    for _ in range(20):
        tokens = torch.randint(0, M, (1, S, K), generator=g)
        parents = torch.randint(0, K, (1, S, K), generator=g).to(torch.int32)
        scores = torch.sort(torch.rand(1, S, K, generator=g), dim=2, descending=True)[0]
        n = int(torch.randint(1, M + 1, (1,), generator=g))
        b = Beams(tokens, parents, scores, torch.zeros(1, S, K, M))
        for (row, _), (idx, sc) in zip(b.paths()[0], b.n_best([n])[0]):
            assert idx == greedy_search(torch.nn.functional.one_hot(torch.tensor(row), M).float(), n)
        assert [sc for _, sc in b.n_best([n])[0]] == scores[0, -1].tolist()


def test_summary_keeps_its_four_field_form():
    s = Summary(torch.zeros(1, 2, 3), None, torch.tensor([[0, -1]], dtype=torch.int32), torch.tensor([1], dtype=torch.int32))
    assert s.beams is None and s.to_lists() == [[0]]
    probs, loss, idx, cnt = s[:4]
    assert loss is None and idx.shape == (1, 2)
