"""CPU: the options of samples without replacement (the stochastic beam) are checked by MMBiDAF.summarize and Summarizer before any
device work; the host statement of the child key; Inclusion's probabilities and weights on hand-built tensors; the C-ABI entry point."""
import math

import numpy as np
import pytest
import torch

from mmbidaf_b200 import ops
from mmbidaf_b200.decode import truncated_key
from mmbidaf_b200.summarize import Inclusion, Summarizer, check_options
from mmbidaf_b200.synth import make_batch

BAD = [dict(replacement=False), dict(replacement=False, num_samples=0), dict(replacement=False, num_samples=9),
       dict(replacement=False, num_samples=True), dict(replacement=False, num_samples=2.0),
       dict(replacement=False, num_samples=2, top_k=3), dict(replacement=False, num_samples=2, top_k=1),
       dict(replacement=False, num_samples=2, top_p=0.9), dict(replacement=False, num_samples=2, top_p=True),
       dict(replacement=False, num_samples=2, beam_width=2), dict(replacement=False, num_samples=2, temperature=0),
       dict(replacement=False, num_samples=2, temperature=math.nan), dict(replacement=False, num_samples=2, seed=1.5),
       dict(replacement=0, num_samples=2), dict(replacement="no", num_samples=2), dict(replacement=None)]


@pytest.fixture(scope="module")
def model():
    from mmbidaf_b200.models import MMBiDAF
    return MMBiDAF(100, 300, 128, 1000, torch.device("cpu"), drop_prob=0.0, max_transcript_length=64)


@pytest.mark.parametrize("kw", BAD)
def test_summarize_rejects_bad_options_before_device_work(model, kw):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    before = ops.launch_count
    with pytest.raises(ValueError, match="replacement|num_samples|temperature|top_k|top_p|seed|beam_width"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, **kw)
    assert ops.launch_count == before
    summarizer = Summarizer(model)
    with pytest.raises(ValueError, match="replacement|num_samples|temperature|top_k|top_p|seed|beam_width"):
        summarizer(b, **kw)
    assert summarizer.buckets == {}


def test_targets_are_rejected(model):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    with pytest.raises(ValueError, match="targets"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, num_samples=2,
                        replacement=False)
    with pytest.raises(ValueError, match="targets"):
        Summarizer(model)(b, with_targets=True, num_samples=2, replacement=False)


def test_good_options_pass():
    for k in range(1, 9):
        for t in (0.1, 1, 2.5):
            for seed in (None, 0, 1 << 70):
                for nr, ms in ((False, 0), (True, 3)):
                    check_options("summarize", False, None, nr, ms, k, t, 0, seed, 1.0, False)
    check_options("summarize", False, None, False, 0, 64, 1.0, 0, None, 1.0, True)     # with replacement: up to 64, as before


def _uniform_ends():
    """The smallest and largest uniform of the sampled rule, ((h >> 9) + 0.5) 2^-23, and their Gumbel perturbations in fp32."""
    u = np.array([0.5 * 2.0 ** -23, ((1 << 23) - 1 + 0.5) * 2.0 ** -23], dtype=np.float32)
    assert u[0] == np.float32(2.0 ** -24) and u[1] == np.float32(1 - 2.0 ** -24)
    return -np.log(-np.log(u))


def test_key_of_the_largest_child_is_the_parent_key():
    for kp in (0.0, -1.5, 3.25, -40.0):
        for z in (-3.0, 0.0, 2.5, 17.0):
            assert truncated_key(kp, z, z) == np.float32(kp)


def test_key_is_monotone_and_at_most_the_parent_key():
    for kp in (0.0, -2.0, 5.0):
        z = np.float32(1.25)
        g = np.sort(np.concatenate([z - np.geomspace(1e-6, 60, 400, dtype=np.float32), [z]])).astype(np.float32)
        k = truncated_key(kp, g, z)
        assert np.all(np.isfinite(k))
        assert np.all(np.diff(k) >= 0)                     # monotone in G
        assert np.all(k <= np.float32(kp))


def test_key_is_finite_at_both_ends_of_the_uniform():
    gum = _uniform_ends()
    assert np.all(np.isfinite(gum))
    for phi in (0.0, -5.0, -80.0):
        g = np.float32(phi) + gum.astype(np.float32)
        z = g.max()
        for kp in (0.0, -3.0, 12.0):
            k = truncated_key(kp, g, z)
            assert np.all(np.isfinite(k)) and k[np.argmax(g)] == np.float32(kp)


def test_inclusion_probabilities_and_weights():
    ninf = -math.inf
    logq = torch.tensor([[math.log(0.5), math.log(0.3), math.log(0.2)],
                         [math.log(0.6), math.log(0.1), ninf],
                         [-1.0, -2.0, -3.0]], dtype=torch.float32)
    keys = torch.tensor([[0.0, -0.5, -1.0], [0.0, -2.0, ninf], [0.5, -0.1, -0.7]])
    thr = torch.tensor([ninf, ninf, -1.5])
    inc = Inclusion(logq, keys, thr)
    p = inc.probabilities()
    assert p.dtype == torch.float64
    assert torch.equal(p[0], torch.ones(3, dtype=torch.float64))                 # kappa = -inf: every sequence is in
    assert p[1].tolist() == [1.0, 1.0, 0.0]                                       # an empty slot: 0
    want = 1 - torch.exp(-torch.exp(logq[2].double() - thr[2].double()))
    assert torch.allclose(p[2], want, rtol=1e-12, atol=0)
    w = inc.weights(normalise=False)
    assert torch.allclose(w[0], torch.exp(logq[0].double()), rtol=0, atol=0)     # kappa = -inf: weight = exp(logq)
    assert w[1, 2] == 0 and torch.allclose(w[1, :2], torch.exp(logq[1, :2].double()))
    assert torch.allclose(w[2], torch.exp(logq[2].double()) / want, rtol=1e-12, atol=0)
    wn = inc.weights()
    assert torch.allclose(wn.sum(1), torch.ones(3, dtype=torch.float64), rtol=1e-12, atol=0)
    assert wn[1, 2] == 0


def test_capi_declares_the_entry_point():
    import os
    import re
    from conftest import ROOT
    from mmbidaf_b200 import _lib
    text = open(os.path.join(ROOT, "include", "mmbidaf_b200.h")).read()
    assert re.search(r"MMB_API\s+int\s+mmb_decoder_beam_sample_fused\s*\(", text)
    assert "mmb_decoder_beam_sample_fused" in _lib.SIGNATURES
