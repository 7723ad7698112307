"""CPU: the options of sampled summaries are checked by MMBiDAF.summarize and Summarizer before any device work, and the host side
of a sampled Summary -- logp, the likeliest sample and Samples.summaries -- on hand-built tensors."""
import math

import pytest
import torch

from mmbidaf_b200 import ops
from mmbidaf_b200.summarize import Samples, Summarizer, best_sample, check_options, sample_logp
from mmbidaf_b200.synth import make_batch

BAD = [dict(num_samples=0), dict(num_samples=65), dict(num_samples=True), dict(num_samples=2.0), dict(num_samples="4"),
       dict(num_samples=2, temperature=0), dict(num_samples=2, temperature=-1.0), dict(num_samples=2, temperature=math.inf),
       dict(num_samples=2, temperature=math.nan), dict(num_samples=2, temperature=True), dict(num_samples=2, temperature="hot"),
       dict(num_samples=2, top_k=-1), dict(num_samples=2, top_k=9), dict(num_samples=2, top_k=2.0), dict(num_samples=2, seed=1.5),
       dict(num_samples=2, seed=True), dict(num_samples=2, beam_width=2), dict(temperature=0.5), dict(top_k=3), dict(seed=1)]


@pytest.fixture(scope="module")
def model():
    from mmbidaf_b200.models import MMBiDAF
    return MMBiDAF(100, 300, 128, 1000, torch.device("cpu"), drop_prob=0.0, max_transcript_length=64)


@pytest.mark.parametrize("kw", BAD)
def test_summarize_rejects_bad_sampling_options_before_device_work(model, kw):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    before = ops.launch_count
    with pytest.raises(ValueError, match="num_samples|temperature|top_k|seed"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, **kw)
    assert ops.launch_count == before
    summarizer = Summarizer(model)
    with pytest.raises(ValueError, match="num_samples|temperature|top_k|seed"):
        summarizer(b, **kw)
    assert summarizer.buckets == {}


def test_sampling_with_targets_is_rejected(model):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    with pytest.raises(ValueError, match="targets"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, num_samples=2)
    with pytest.raises(ValueError, match="targets"):
        Summarizer(model)(b, with_targets=True, num_samples=2)


def test_good_options_pass():
    for n in (1, 64):
        for t in (0.1, 1, 2.5):
            for k in (0, 1, 8):
                for seed in (None, 0, -3, 1 << 70):
                    check_options("summarize", False, None, True, 3, n, t, k, seed)


def test_logp_best_sample_and_summaries():
    # B = 2 videos, N = 3 samples, S = 4 steps, M = 5 rows; video 0's EOS row is 3, video 1's is 1
    torch.manual_seed(0)
    probs = torch.softmax(torch.randn(2, 3, 4, 5), -1)
    tokens = torch.tensor([[[0, 2, 3, 1], [4, 3, 3, 3], [2, 2, 2, 2]],
                           [[1, 0, 0, 0], [0, 1, 1, 1], [3, 0, 1, 0]]])
    lens = torch.tensor([4, 2], dtype=torch.int32)
    logp = sample_logp(probs, tokens, lens)
    lp = lambda v, n, steps: sum(math.log(float(probs[v, n, s, tokens[v, n, s]])) for s in steps)
    want = [[lp(0, 0, range(3)), lp(0, 1, range(2)), lp(0, 2, range(4))],
            [lp(1, 0, range(1)), lp(1, 1, range(2)), lp(1, 2, range(3))]]
    assert torch.allclose(logp.double(), torch.tensor(want, dtype=torch.float64), rtol=1e-6, atol=0)
    smp = Samples(tokens, probs, logp)
    got = logp.tolist()
    assert smp.summaries(lens) == [[([0, 2], got[0][0]), ([], got[0][1]), ([2, 2, 2, 2], got[0][2])],
                                   [([], got[1][0]), ([0], got[1][1]), ([0], got[1][2])]]
    # the greedy selection of every sample's tokens, as ops.greedy_select gives it, and the likeliest sample of each video
    sel = torch.full((6, 4), -1, dtype=torch.int32)
    cnt = torch.zeros(6, dtype=torch.int32)
    for r, (chosen, _) in enumerate(x for per in smp.summaries(lens) for x in per):
        sel[r, :len(chosen)] = torch.tensor(chosen, dtype=torch.int32)
        cnt[r] = len(chosen)
    dist, idx, count = best_sample(smp, sel, cnt)
    for v in range(2):
        n = max(range(3), key=lambda k: (float(logp[v, k]), -k))
        assert torch.equal(dist[v], probs[v, n]) and torch.equal(idx[v], sel[v * 3 + n]) and int(count[v]) == int(cnt[v * 3 + n])


def test_ties_go_to_the_lower_sample():
    probs = torch.full((1, 3, 2, 2), 0.5)
    tokens = torch.tensor([[[0, 1], [1, 0], [0, 0]]])
    logp = sample_logp(probs, tokens, torch.tensor([2], dtype=torch.int32))
    assert logp[0, 0] == logp[0, 2]                        # n = 0 stops at its EOS pick (row 1), n = 2 has none
    smp = Samples(tokens, probs, torch.tensor([[-1.0, -3.0, -1.0]]))
    _, idx, _ = best_sample(smp, torch.arange(6, dtype=torch.int32).view(3, 2), torch.ones(3, dtype=torch.int32))
    assert idx.tolist() == [[0, 1]]

