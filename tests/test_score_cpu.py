"""CPU: summary scoring -- the candidate rows of host lists (summarize.candidate_tokens), its errors, the shared logp rule
(summarize.path_logp, the rule of Samples.logp and Scores.logp) and the C-ABI entry point."""
import math
import os
import re

import pytest
import torch

from conftest import ROOT
from mmbidaf_b200.summarize import candidate_tokens, path_logp, sample_logp


def test_rows_eos_placement_and_padding():
    # video 0: EOS row 4; video 1: EOS row 2; video 2: EOS row 6, no candidate
    tokens, valid = candidate_tokens([[[0, 3], [], [1, 2, 3, 0]], [[1]], []], [5, 3, 7], 4)
    assert tokens.dtype == torch.int64 and tokens.shape == (3, 3, 4)
    assert valid.dtype == torch.bool and valid.tolist() == [[True, True, True], [True, False, False], [False, False, False]]
    assert tokens[0].tolist() == [[0, 3, 4, 4], [4, 4, 4, 4], [1, 2, 3, 0]]     # the last: exactly S indices, no EOS
    assert tokens[1, 0].tolist() == [1, 2, 2, 2]
    assert (tokens[1, 1:] == 2).all() and (tokens[2] == 6).all()               # padding rows: EOS throughout


def test_pairs_tensor_lengths_and_integer_types():
    import numpy as np
    a, va = candidate_tokens([[([2, 0], -1.5), (np.int64(1),)]], torch.tensor([4], dtype=torch.int32), 3)
    assert a.tolist() == [[[2, 0, 3], [1, 3, 3]]] and va.all()


@pytest.mark.parametrize("cands,lens,steps", [
    ([[[0, 4]]], [5], 4),               # index == eos
    ([[[-1]]], [5], 4),                 # negative
    ([[[7]]], [5], 4),                  # past eos
    ([[[0, 1, 2]]], [9], 2),            # more indices than steps
    ([[[0]] * 65], [5], 4),             # more than 64 candidates
    ([[], []], [5, 5], 4),              # no candidate at all
    ([], [], 4),
    ([[[0]]], [5, 6], 4),               # lengths for another batch
    ([[[0.5]]], [5], 4),                # not an index
    ([[[True]]], [5], 4),
    ([[[0]]], [5], 0),                  # no steps
])
def test_errors(cands, lens, steps):
    with pytest.raises(ValueError, match="candidate_tokens"):
        candidate_tokens(cands, lens, steps)


def test_shared_logp_rule_on_hand_made_rows():
    step_p = torch.tensor([[[0.5, 0.25, 0.125, 0.5], [0.1, 0.2, 0.3, 0.4]],
                           [[0.9, 0.8, 0.7, 0.6], [1.0, 0.5, 0.5, 0.5]]])
    tokens = torch.tensor([[[1, 4, 4, 0], [1, 2, 3, 1]],          # video 0, EOS 4: stops after step 1; no EOS: all four
                           [[2, 0, 2, 2], [2, 2, 2, 2]]])         # video 1, EOS 2: the first step is the EOS
    lens = torch.tensor([5, 3], dtype=torch.int32)
    got = path_logp(step_p, tokens, lens)
    want = [[math.log(0.5) + math.log(0.25), sum(math.log(x) for x in (0.1, 0.2, 0.3, 0.4))],
            [math.log(0.9), math.log(1.0)]]
    assert torch.allclose(got.double(), torch.tensor(want, dtype=torch.float64), rtol=1e-6, atol=1e-7)
    # Samples.logp is the same rule over the gathered rows, unchanged bit for bit
    M = 6
    probs = torch.rand(2, 2, 4, M, generator=torch.Generator().manual_seed(3))
    tok = torch.randint(0, M, (2, 2, 4), generator=torch.Generator().manual_seed(4))
    tok[0, 0, 2] = 4
    gathered = probs.gather(3, tok.unsqueeze(3)).squeeze(3)
    assert torch.equal(sample_logp(probs, tok, lens), path_logp(gathered, tok, lens))
    lp = torch.log(gathered)
    hit = (tok == (lens.long() - 1).view(-1, 1, 1)).long()
    assert torch.equal(sample_logp(probs, tok, lens), torch.where((hit.cumsum(2) - hit) > 0, torch.zeros_like(lp), lp).sum(2))


def test_zero_step_probability_gives_minus_infinity():
    got = path_logp(torch.tensor([[[0.5, 0.0]]]), torch.tensor([[[1, 3]]]), torch.tensor([4], dtype=torch.int32))
    assert got.item() == -math.inf


def test_entry_point_is_declared_and_bound():
    from mmbidaf_b200 import _lib
    text = open(os.path.join(ROOT, "include", "mmbidaf_b200.h")).read()
    assert re.search(r"MMB_API\s+int\s+mmb_decoder_forced_fused\s*\(", text)
    assert "mmb_decoder_forced_fused" in _lib.SIGNATURES
