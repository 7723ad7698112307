"""CPU: the options of constrained summaries (no_repeat, min_sentences) are checked by MMBiDAF.summarize and Summarizer before any
device work -- here on a machine without one, so a check that came after a launch would fail differently."""
import pytest
import torch

from mmbidaf_b200 import ops
from mmbidaf_b200.summarize import Summarizer, check_options
from mmbidaf_b200.synth import make_batch

BAD = [dict(no_repeat=1), dict(no_repeat=None), dict(no_repeat="yes"), dict(min_sentences=-1), dict(min_sentences=2.0),
       dict(min_sentences=True), dict(min_sentences=None)]


@pytest.fixture(scope="module")
def model():
    from mmbidaf_b200.models import MMBiDAF
    return MMBiDAF(100, 300, 128, 1000, torch.device("cpu"), drop_prob=0.0, max_transcript_length=64)


@pytest.mark.parametrize("kw", BAD)
@pytest.mark.parametrize("beam_width", [None, 2])
def test_summarize_rejects_bad_options_before_device_work(model, kw, beam_width):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    before = ops.launch_count
    with pytest.raises(ValueError, match="no_repeat|min_sentences"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, beam_width=beam_width, **kw)
    assert ops.launch_count == before


@pytest.mark.parametrize("kw", [dict(no_repeat=True), dict(min_sentences=1), dict(no_repeat=True, min_sentences=3)])
def test_constraints_with_targets_are_rejected(model, kw):
    b = make_batch(2, 11, 13, 3, 4, seed=1)
    with pytest.raises(ValueError, match="targets"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, **kw)
    summarizer = Summarizer(model)
    with pytest.raises(ValueError, match="targets"):
        summarizer(b, with_targets=True, **kw)
    assert summarizer.buckets == {}


@pytest.mark.parametrize("kw", BAD + [dict(beam_width=0), dict(beam_width=9), dict(beam_width=True)])
def test_summarizer_rejects_bad_options_before_capture(model, kw):
    summarizer = Summarizer(model)
    with pytest.raises(ValueError, match="no_repeat|min_sentences|beam_width"):
        summarizer(make_batch(2, 11, 13, 3, 4, seed=1), **kw)
    assert summarizer.buckets == {}


def test_good_options_pass():
    for w in (None, 1, 8):
        for nr in (False, True):
            for ms in (0, 1, 50):
                check_options("summarize", False, w, nr, ms)
    check_options("summarize", True, None, False, 0)       # targets without constraints: the eval loss of the greedy roll-out
