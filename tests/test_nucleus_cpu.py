"""CPU: the top_p option of sampled summaries is checked by MMBiDAF.summarize and Summarizer before any device work, and the nucleus
rule (include/mmbidaf_b200.h at mmb_decoder_sample_nucleus_fused) as decode.nucleus states it on the host, on hand-built rows."""
import math

import numpy as np
import pytest
import torch

from mmbidaf_b200 import ops
from mmbidaf_b200.decode import nucleus
from mmbidaf_b200.summarize import Summarizer, check_options
from mmbidaf_b200.synth import make_batch

BAD = [dict(num_samples=2, top_p=0), dict(num_samples=2, top_p=0.0), dict(num_samples=2, top_p=-0.1), dict(num_samples=2, top_p=1.5),
       dict(num_samples=2, top_p=math.nan), dict(num_samples=2, top_p=math.inf), dict(num_samples=2, top_p=True),
       dict(num_samples=2, top_p="0.9"), dict(num_samples=2, top_p=1e-50), dict(top_p=0.9), dict(top_p=0.9, beam_width=2),
       dict(top_p=True), dict(top_p=math.nan)]


@pytest.fixture(scope="module")
def model():
    from mmbidaf_b200.models import MMBiDAF
    return MMBiDAF(100, 300, 128, 1000, torch.device("cpu"), drop_prob=0.0, max_transcript_length=64)


@pytest.mark.parametrize("kw", BAD)
def test_summarize_rejects_bad_top_p_before_device_work(model, kw):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    before = ops.launch_count
    with pytest.raises(ValueError, match="top_p"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, **kw)
    assert ops.launch_count == before
    summarizer = Summarizer(model)
    with pytest.raises(ValueError, match="top_p"):
        summarizer(b, **kw)
    assert summarizer.buckets == {}


def test_top_p_with_targets_is_rejected(model):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    with pytest.raises(ValueError, match="top_p"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, top_p=0.9)
    with pytest.raises(ValueError, match="top_p"):
        Summarizer(model)(b, with_targets=True, top_p=0.9)
    with pytest.raises(ValueError, match="targets"):
        Summarizer(model)(b, with_targets=True, num_samples=2, top_p=0.9)


def test_the_ops_check_rejects_bad_top_p():
    for top_p in (0, -0.1, 1.5, math.nan, math.inf, True, False, "0.9", None, 1e-50):
        with pytest.raises(ValueError, match="top_p"):
            ops.check_sampling("sample_pick", 2, 1.0, 0, top_p)


def test_good_options_pass():
    for top_p in (1e-30, 0.3, 0.9, 1 - 1e-9, 1, 1.0):
        for k in (0, 3, 8):
            check_options("summarize", False, None, True, 3, 4, 0.7, k, 5, top_p)
            ops.check_sampling("sample_pick", 4, 0.7, k, top_p)
    check_options("summarize", False, 2, False, 0, None, 1.0, 0, None, 1.0)     # the default is no option at all


def _p(*xs):
    return np.array(xs, dtype=np.float32)


def test_equality_at_the_boundary_is_included():
    p = _p(0.5, 0.25, 0.25)
    assert nucleus(p, top_p=0.5) == [0]            # 2^24 q_0 == P Q exactly
    assert nucleus(p, top_p=0.75) == [0, 1]
    assert nucleus(p, top_p=0.7500001) == [0, 1, 2]
    assert nucleus(p, top_p=0.4999999) == [0]
    assert nucleus(p, top_p=0.5000001) == [0, 1]


def test_ties_at_the_boundary_go_by_m():
    p = _p(0.25, 0.25, 0.25, 0.25)
    assert nucleus(p, top_p=0.5) == [0, 1]
    assert nucleus(p, top_p=0.51) == [0, 1, 2]
    assert nucleus(p, eligible=[0, 1, 1, 1], top_p=0.5) == [1, 2]          # need = 1.5 q: two ties
    q = _p(0.1, 0.3, 0.1, 0.3, 0.1, 0.1)
    assert nucleus(q, top_p=0.6) == [1, 3]
    assert nucleus(q, top_p=0.61) == [1, 3, 0]
    assert nucleus(q, top_p=0.81) == [1, 3, 0, 2, 4]


@pytest.mark.parametrize("M", [1, 2, 409, 4096])
@pytest.mark.parametrize("top_p", [0.05, 0.5, 0.9, 0.999])
def test_uniform_rows(M, top_p):
    p = np.full(M, np.float32(1.0) / np.float32(M), dtype=np.float32)
    P = int(np.rint(float(np.float32(top_p)) * 2 ** 24))
    n = max(1, -(-P * M // 2 ** 24))                                        # n q 2^24 >= P M q
    assert nucleus(p, top_p=top_p) == list(range(n))
    assert nucleus(torch.from_numpy(p), top_p=top_p) == list(range(n))      # a tensor row too


def test_rows_with_zeros():
    p = _p(0.0, 0.5, 0.0, 0.5)
    assert nucleus(p, top_p=0.9999) == [1, 3]                               # q = 0 is never needed
    assert nucleus(p) == [1, 3, 0, 2]                                        # top_p = 1: no cut, the zeros stay candidates
    assert nucleus(_p(0.0, 1.0, 0.0), eligible=[1, 0, 1], top_p=0.9) == [0]   # Q = 0: n = 1, the first candidate
    assert nucleus(_p(1e-8, 1.0, 2e-8), eligible=[1, 0, 1], top_p=0.9) == [2]  # q = 0 below 2^-24, the likeliest still first
    assert nucleus(_p(0.3, 0.7), eligible=[0, 0], top_p=0.5) == []            # no candidate


def test_combination_with_top_k():
    p = _p(0.1, 0.4, 0.3, 0.2)
    assert nucleus(p, top_k=2) == [1, 2]
    assert nucleus(p, top_k=2, top_p=0.5) == [1]                             # 0.4 >= 0.5 (0.4 + 0.3)
    assert nucleus(p, top_k=2, top_p=0.6) == [1, 2]                          # 0.4 <  0.6 (0.4 + 0.3)
    assert nucleus(p, top_k=3, top_p=0.6) == [1, 2]                          # 0.7 >= 0.6 (0.9)
    assert nucleus(p, top_k=3, top_p=0.8) == [1, 2, 3]
    assert nucleus(p, top_k=1, top_p=0.01) == [1]
    assert nucleus(p, eligible=[1, 0, 1, 1], top_k=2, top_p=0.6) == [2]      # 0.3 >= 0.6 (0.3 + 0.2): the cut follows the constraint
    assert nucleus(p, eligible=[1, 0, 1, 1], top_k=2, top_p=0.7) == [2, 3]


def test_p_rounds_half_to_even():
    """P = rint(top_p 2^24): at top_p 2^24 = 2^22 + 1/2 it is 2^22 (even), at 2^22 + 3/2 it is 2^22 + 2.  Four equal masses give
    n = 1 exactly when P <= 2^22."""
    p = np.full(4, np.float32(2.0 ** -24), dtype=np.float32)
    lo, hi = np.float32(0.25 + 2.0 ** -25), np.float32(0.25 + 3 * 2.0 ** -25)
    assert float(lo) * 2 ** 24 == 2 ** 22 + 0.5 and float(hi) * 2 ** 24 == 2 ** 22 + 1.5
    assert nucleus(p, top_p=float(lo)) == [0]
    assert nucleus(p, top_p=float(hi)) == [0, 1]
    assert nucleus(p, top_p=0.25) == [0]


def test_the_masses_are_exact():
    """q = floor(p 2^24) from the fp32 p: the largest fp32 below 1 has q = 2^24 - 1, p = 2^-25 has q = 0."""
    big = np.nextafter(np.float32(1.0), np.float32(0.0))
    p = _p(float(big), 2.0 ** -24, 2.0 ** -25)
    # Q = 2^24 - 1 + 1 + 0 = 2^24: need = P, so n = 1 while P <= 2^24 - 1
    assert nucleus(p, top_p=float(big)) == [0]
    assert nucleus(p, top_p=1.0) == [0, 1, 2]
