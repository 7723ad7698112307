"""GPU: summarisation -- MMBiDAF.summarize (the greedy roll-out as one cluster kernel, or the chunk cut for long lectures) against
the eval-mode forward + decode.get_generated_indices, the device-side greedy selection, graph replay (Summarizer), and the summaries
of a two-rank data-parallel job gathered on rank 0."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import load_golden
from mmbidaf_b200.decode import get_generated_indices, greedy_search
from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu


def _model(m, seed=224):
    from mmbidaf_b200.models import MMBiDAF
    params = O.make_params(100, 300, 128, 1000, m, seed=seed)
    model = MMBiDAF(100, 300, 128, 1000, torch.device("cuda"), drop_prob=0.0, max_transcript_length=m)
    model.load_state_dict(params)
    return model.cuda()


def _forward_eval(model, b, steps):
    model.eval()
    with torch.no_grad():
        return model(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, b.targets, b.target_len, steps)


def _summarize(model, b, steps, targets):
    return model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, steps,
                           targets=b.targets if targets else None)


@pytest.fixture
def tier(request):
    import mmbidaf_b200
    mmbidaf_b200.set_precision(request.param)
    yield request.param
    mmbidaf_b200.set_precision("fp32")


def _batch(B, lt=37, la=45, li=7, t_dec=16, seed=5):
    b = make_batch(B, lt, la, li, t_dec, seed=seed + B)
    if B > 1:                                              # a two-row transcript: one sentence and the EOS row
        n = 2
        b.text[1, n - 1:] = 0
        b.text[1, n - 1] = -1.0
        b.text_len[1] = n
        b.targets[1] = 0
        b.targets[1, 0, 0] = float(n - 1)
    return b


def _check(model, b, steps, targets):
    out, loss = _forward_eval(model, b, steps)
    model.train()                                          # summarize gives the caller's training flag back
    s = _summarize(model, b, steps, targets)
    assert model.training
    assert s.out_distributions.shape == out.shape
    assert torch.equal(s.out_distributions, out)
    if targets:
        assert torch.equal(s.loss, loss)
    else:
        assert s.loss is None
    want = get_generated_indices(out, b.text_len)
    assert s.to_lists() == want
    assert s.indices.dtype == torch.int32 and s.counts.dtype == torch.int32
    assert s.counts.cpu().tolist() == [len(w) for w in want]
    return want


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 20, 21, 32])
@pytest.mark.parametrize("targets", [True, False])
def test_summarize_equals_eval_forward(tier, B, targets):
    model = _model(64)                                     # M = 64 > Lt = 37 (odd)
    b = _batch(B).to("cuda")
    for steps in (1, 16):
        _check(model, b, steps, targets)


def test_summary_of_a_video_whose_first_pick_is_its_eos_row():
    model = _model(64)
    b = _batch(3).to("cuda")
    k = b.text_len[2] - 1                                  # video 2's EOS row: every video whose mask covers it picks it
    with torch.no_grad():
        model.multimodal_att_decoder.out.bias[k] += 60.0
    want = _check(model, b, 16, True)
    assert want[2] == []


def test_long_lecture_side_of_the_rule_equals_forward():
    from mmbidaf_b200 import ops
    model = _model(700)
    b = make_batch(32, 700, 60, 6, 6, seed=41).to("cuda")
    assert ops.decoder_cut(32, 700) == "chunks"
    for targets in (True, False):
        _check(model, b, 6, targets)


def test_full_config5_summaries_have_the_long_lecture_properties():
    m = 4096
    model = _model(m)
    batch = make_batch(16, 4096, 4096, 2048, 16, seed=32)
    b = batch.to("cuda")
    s = _summarize(model, b, 16, True)
    out = s.out_distributions
    assert out.shape == (16, 16, m) and torch.isfinite(out).all() and torch.isfinite(s.loss)
    assert (out.sum(dim=2) - 1).abs().max() < 1e-4
    lens = torch.tensor(batch.text_len, device="cuda")
    beyond = torch.arange(m, device="cuda").view(1, 1, m) >= lens.view(-1, 1, 1)
    assert (out.masked_select(beyond.expand_as(out)) == 0).all()
    picks = s.to_lists()
    assert picks == get_generated_indices(out, batch.text_len)
    assert all(0 <= k < n - 1 for ks, n in zip(picks, batch.text_len) for k in ks)


def _select(argmax, lengths):
    from mmbidaf_b200 import ops
    sel, count = ops.greedy_select(argmax.cuda(), torch.tensor(lengths, dtype=torch.int32, device="cuda"))
    sel, count = sel.cpu(), count.cpu()
    got = [sel[b, :int(count[b])].tolist() for b in range(len(lengths))]
    assert all((sel[b, int(count[b]):] == -1).all() for b in range(len(lengths)))
    return got


def test_greedy_select_matches_greedy_search_on_random_tables():
    g = torch.Generator().manual_seed(9)
    for B, S in ((1, 1), (5, 16), (130, 7), (33, 40)):
        lengths = torch.randint(1, 20, (B,), generator=g).tolist()
        # indices below, at and beyond the EOS row len - 1
        argmax = torch.stack([torch.randint(0, n + 3, (S,), generator=g) for n in lengths])
        M = int(argmax.max()) + 1
        want = [greedy_search(torch.nn.functional.one_hot(argmax[b], M).float(), lengths[b]) for b in range(B)]
        assert _select(argmax, lengths) == want


def test_greedy_select_matches_the_reference_fixtures():
    for case in load_golden("greedy_search.pt")["cases"]:
        argmax = case["dist"].cuda().argmax(dim=2)
        assert _select(argmax, case["lengths"]) == case["indices"]


def test_summarizer_replays_equal_eager_summarize():
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    summarizer = Summarizer(model)
    batches = [make_batch(4, 37, 45, 7, 12, seed=s).to("cuda") for s in (1, 2, 3)]
    assert len({tuple(b.text_len) for b in batches}) == 3                   # one bucket, three sets of lengths
    for with_targets in (False, True):
        for b in batches:
            got = summarizer(b, with_targets=with_targets)
            got = [None if t is None else t.clone() for t in got]
            want = _summarize(model, b, b.max_dec_len, with_targets)
            for g, w in zip(got, want):
                assert (g is None and w is None) or torch.equal(g, w)
    assert len(summarizer.buckets) == 2                                     # with and without targets
    other = make_batch(4, 29, 45, 7, 12, seed=4).to("cuda")                 # another text width: a new bucket
    got = summarizer(other)
    assert len(summarizer.buckets) == 3
    assert torch.equal(got.out_distributions, _summarize(model, other, other.max_dec_len, False).out_distributions)
    with torch.no_grad():                                                   # an optimiser-style in-place update
        model.multimodal_att_decoder.out.weight.mul_(1.5)
        model.multimodal_att_decoder.W2.weight.add_(0.01)
        model.text_enc.rnn.weight_hh_l0.mul_(0.9)
    got = summarizer(batches[0])
    want = _summarize(model, batches[0], batches[0].max_dec_len, False)
    assert torch.equal(got.out_distributions, want.out_distributions) and torch.equal(got.indices, want.indices)


def _ddp_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from mmbidaf_b200.summarize import gather_summaries
    from mmbidaf_b200.trainer import shard_batch
    model = _model(64)
    shard = shard_batch(_batch(5), rank, world).to("cuda")
    out[rank] = gather_summaries(_summarize(model, shard, 12, False))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_gathered_summaries_equal_the_single_process_summaries():
    world, port = 2, 29500 + os.getpid() % 2000
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_ddp_worker, args=(world, port, out), nprocs=world, join=True)
        got = {r: out[r] for r in range(world)}
    want = _summarize(_model(64), _batch(5).to("cuda"), 12, False).to_lists()
    assert got[1] is None and got[0] == want
