"""GPU: beam-search summarisation -- the beam roll-out as one cluster kernel (mmb_decoder_beam_fused) against a host loop of the
fused step kernel that applies the same rule, width 1 against the greedy summary, the n-best lists, graph replay (Summarizer) and
the errors."""
import math

import pytest
import torch

from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu

EMPTY, LIVE, DONE = 0, 1, 2


def _model(m, seed=224):
    from mmbidaf_b200.models import MMBiDAF
    params = O.make_params(100, 300, 128, 1000, m, seed=seed)
    model = MMBiDAF(100, 300, 128, 1000, torch.device("cuda"), drop_prob=0.0, max_transcript_length=m)
    model.load_state_dict(params)
    return model.cuda()


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


def _summarize(model, b, steps, beam_width=None):
    return model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, steps, beam_width=beam_width)


def _decoder_inputs(model, b):
    """What summarize hands the decoder: (emb_text, h0, enc_a, enc_i, mask, text_len int32)."""
    from mmbidaf_b200.layers.encoding import length_plan
    model.eval()
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    return b.text, h0, enc_a, enc_i, mask, length_plan(b.text_len, b.text.device).len_i32.clone()


def _reference(dec, emb, h0, enc_a, enc_i, mask, text_len, steps, K):
    """The beam rule as a host loop: per step, the fused step kernel once per slot on all B videos, candidates score + log(p) in
    fp32 on the device, stable sorts in reverse key order, then the state gathered by parent."""
    from mmbidaf_b200 import ops
    with torch.no_grad():
        seq = dec._sequence(enc_a, enc_i)["seq"]
        B, Lt, H, M = seq.B, seq.Lt, seq.H, seq.M
        dev = emb.device
        mask_u8 = ops._u8(mask)
        rows = torch.arange(B, device=dev)
        eos = text_len.long() - 1
        h = torch.zeros(B, K, H, device=dev)
        h[:, 0] = h0.reshape(B, H)
        cell, cov = torch.zeros(B, K, H, device=dev), torch.zeros(B, K, Lt, device=dev)
        tok = torch.full((B, K), -1, dtype=torch.long, device=dev)
        score = torch.full((B, K), -math.inf, device=dev)
        score[:, 0] = 0
        stat = torch.full((B, K), EMPTY, dtype=torch.long, device=dev)
        stat[:, 0] = LIVE
        T, P, S_, R = [], [], [], []
        slot = torch.arange(K, device=dev).view(1, K, 1).expand(B, K, M)
        sent_of = torch.arange(M, device=dev).view(1, 1, M).expand(B, K, M)
        for s in range(steps):
            p = torch.zeros(B, K, M, device=dev)
            hn, cn, vn = torch.zeros_like(h), torch.zeros_like(cell), torch.zeros_like(cov)
            for k in range(K):
                sent = emb.new_zeros(B, emb.shape[2]) if s == 0 else emb[rows, tok[:, k].clamp(0, Lt - 1)]
                out = ops.decoder_step_fwd(seq, sent.contiguous(), h[:, k].contiguous(), cell[:, k].contiguous(),
                                           cov[:, k].contiguous(), mask_u8)
                p[:, k], hn[:, k], cn[:, k], vn[:, k] = out[0], out[1], out[2], out[4]
            live = (stat == LIVE).unsqueeze(2) & (p > 0)
            c_score = torch.cat([(score.unsqueeze(2) + torch.log(p)).reshape(B, -1), score], 1)
            c_p = torch.cat([p.reshape(B, -1), torch.ones(B, K, device=dev)], 1)
            c_par = torch.cat([slot.reshape(B, -1), torch.arange(K, device=dev).expand(B, K)], 1)
            c_tok = torch.cat([sent_of.reshape(B, -1), eos.view(B, 1).expand(B, K)], 1)
            c_ok = torch.cat([live.reshape(B, -1), stat == DONE], 1)
            c_carry = torch.cat([torch.zeros(B, K * M, dtype=torch.bool, device=dev), stat == DONE], 1)
            order = torch.arange(c_score.shape[1], device=dev).expand(B, -1)
            for key, desc in ((c_tok, False), (c_par, False), (c_p, True), (c_score, True), (c_ok.to(torch.int8), True)):
                _, idx = torch.sort(key.gather(1, order), dim=1, descending=desc, stable=True)
                order = order.gather(1, idx)
            top = order[:, :K]
            ok = c_ok.gather(1, top)
            par = c_par.gather(1, top)
            t = c_tok.gather(1, top)
            carry = c_carry.gather(1, top)
            sc = c_score.gather(1, top)
            from_live = ok & ~carry
            row = p.gather(1, par.view(B, K, 1).expand(B, K, M)) * from_live.unsqueeze(2)
            T.append(torch.where(ok, t, -1))
            R.append(torch.where(ok, par, -1).to(torch.int32))
            S_.append(torch.where(ok, sc, -math.inf))
            P.append(row)
            g = par.view(B, K, 1)
            h, cell, cov = hn.gather(1, g.expand(B, K, H)), cn.gather(1, g.expand(B, K, H)), vn.gather(1, g.expand(B, K, Lt))
            tok = torch.where(ok, t, -1)
            score = torch.where(ok, sc, -math.inf)
            stat = torch.where(~ok, EMPTY, torch.where(carry | (t == eos.view(B, 1)), DONE, LIVE))
        return torch.stack(T, 1), torch.stack(R, 1), torch.stack(S_, 1), torch.stack(P, 1)


def _check_against_reference(model, b, steps, K):
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    tokens, parents, scores, probs, best, path = dec.beam(emb, h0, enc_a, enc_i, mask, lens, steps, K)
    rt, rp, rs, rprob = _reference(dec, emb, h0, enc_a, enc_i, mask, lens, steps, K)
    assert torch.equal(tokens, rt)
    assert torch.equal(parents, rp)
    assert torch.equal(scores, rs)
    assert torch.equal(probs, rprob)
    # the backtrack: slot 0 after the last step, walked to step 0
    B = tokens.shape[0]
    j = torch.zeros(B, dtype=torch.long, device=tokens.device)
    rows = torch.arange(B, device=tokens.device)
    for s in range(steps - 1, -1, -1):
        assert torch.equal(path[:, s].long(), j)
        assert torch.equal(best[:, s], tokens[rows, s, j])
        j = parents[rows, s, j].long()
    return tokens, parents, scores


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("K", [2, 3, 4, 8])
def test_beam_equals_the_host_loop_of_step_kernels(tier, B, K):
    model = _model(64)                                     # M = 64 > Lt = 37
    b = _batch(B).to("cuda")
    tokens, parents, _ = _check_against_reference(model, b, 16, K)
    if B > 1:                                              # the two-row transcript has two candidates: slots go empty
        assert (parents[1, 0, 2:] == -1).all() and (tokens[1, 0, 2:] == -1).all()


def test_long_lecture_side_of_the_rule_equals_the_host_loop(monkeypatch):
    from mmbidaf_b200 import ops
    model = _model(700)
    b = make_batch(32, 700, 60, 6, 6, seed=41).to("cuda")
    assert ops.decoder_cut(32, 700) == "chunks"            # the beam runs the cluster kernel anyway; so must its reference
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    _check_against_reference(model, b, 6, 3)


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
def test_width_one_is_the_greedy_summary(tier, B):
    from mmbidaf_b200.summarize import Beams
    model = _model(64)
    b = _batch(B).to("cuda")
    greedy = _summarize(model, b, 16)
    beam = _summarize(model, b, 16, beam_width=1)
    assert isinstance(beam.beams, Beams) and greedy.beams is None and beam.loss is None
    assert torch.equal(beam.indices, greedy.indices) and torch.equal(beam.counts, greedy.counts)
    # distributions equal up to each video's first EOS step, zero after
    argmax = greedy.out_distributions.argmax(dim=2).cpu()
    for v in range(B):
        eos = b.text_len[v] - 1
        hits = (argmax[v] == eos).nonzero()
        last = int(hits[0]) if len(hits) else 15
        assert torch.equal(beam.out_distributions[v, :last + 1], greedy.out_distributions[v, :last + 1])
        assert (beam.out_distributions[v, last + 1:] == 0).all()


def test_forced_eos_gives_an_empty_summary_and_a_finished_slot_0():
    model = _model(64)
    b = _batch(3).to("cuda")
    k = b.text_len[2] - 1                                  # video 2's EOS row
    with torch.no_grad():
        model.multimodal_att_decoder.out.bias[k] += 60.0
    s = _summarize(model, b, 16, beam_width=4)
    assert s.to_lists()[2] == []
    tok, par = s.beams.tokens[2].cpu(), s.beams.parents[2].cpu()
    assert int(tok[0, 0]) == k and int(par[0, 0]) == 0     # step 0: slot 0 picks EOS ...
    assert (tok[1:, 0] == k).all() and (par[1:, 0] == 0).all()    # ... and carries it to the end
    assert (s.beams.probs[2, 1:, 0] == 0).all()            # carries have zero rows
    assert s.beams.n_best(b.text_len)[2][0] == ([], float(s.beams.scores[2, -1, 0]))


def test_n_best_rescores_and_is_sorted():
    model = _model(64)
    b = _batch(21).to("cuda")
    K, S = 4, 16
    s = _summarize(model, b, S, beam_width=K)
    bm = s.beams
    paths = bm.paths()
    nbest = bm.n_best(b.text_len)
    probs = bm.probs.cpu()
    tok, par = bm.tokens.cpu(), bm.parents.cpu()
    for v in range(len(paths)):
        assert len(nbest[v]) == len(paths[v]) >= 1
        scores = [sc for _, sc in paths[v]]
        assert scores == sorted(scores, reverse=True)
        rows = [tuple(r) for r, _ in paths[v]]
        assert len(set(rows)) == len(rows)                 # distinct hypotheses
        for j, (row, sc) in enumerate(paths[v]):
            # re-score along the path: the step probability of its token in the row that chose it (a carry's row is zero: it counts
            # as 1), logf on the device, summed in fp32 in step order
            slot, ps = j, []
            for st in range(S - 1, -1, -1):
                ps.append(float(probs[v, st, slot, int(tok[v, st, slot])]))
                slot = int(par[v, st, slot])
            logs = torch.log(torch.tensor([p for p in reversed(ps) if p > 0], device="cuda")).cpu()
            total = torch.zeros((), dtype=torch.float32)
            for x in logs:
                total = total + x
            assert float(total) == sc
    assert nbest[0][0][0] == s.to_lists()[0]


def test_summarizer_replays_equal_eager_beam_summarize():
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    summarizer = Summarizer(model)
    batches = [make_batch(4, 37, 45, 7, 12, seed=s).to("cuda") for s in (1, 2, 3)]
    assert len({tuple(b.text_len) for b in batches}) == 3                   # one bucket, three sets of lengths
    for b in batches:
        got = summarizer(b, beam_width=3)
        got_beams = [t.clone() for t in got.beams]
        got = [t.clone() for t in got[:4] if t is not None]
        want = _summarize(model, b, b.max_dec_len, beam_width=3)
        assert all(torch.equal(g, w) for g, w in zip(got, [t for t in want[:4] if t is not None]))
        assert all(torch.equal(g, w) for g, w in zip(got_beams, want.beams))
    assert len(summarizer.buckets) == 1
    summarizer(batches[0], beam_width=2)                                    # another width: a new bucket
    assert len(summarizer.buckets) == 2
    with torch.no_grad():                                                   # an optimiser-style in-place update
        model.multimodal_att_decoder.out.weight.mul_(1.5)
        model.multimodal_att_decoder.W2.weight.add_(0.01)
    got = summarizer(batches[0], beam_width=3)
    want = _summarize(model, batches[0], batches[0].max_dec_len, beam_width=3)
    assert torch.equal(got.out_distributions, want.out_distributions) and torch.equal(got.beams.scores, want.beams.scores)


def test_widths_launch_at_config3_and_config5_shapes():
    from mmbidaf_b200 import ops
    torch.manual_seed(0)
    D, H, E = 200, 100, 300
    for B, Lt, widths in ((32, 409, range(1, 9)), (16, 4096, range(1, 5))):
        model = _model(Lt)
        dec = model.multimodal_att_decoder
        model.eval()
        enc_a, enc_i = torch.randn(B, Lt, D, device="cuda"), torch.randn(B, Lt, D, device="cuda")
        emb, h0 = torch.randn(B, Lt, E, device="cuda"), torch.randn(B, 1, H, device="cuda")
        lens = torch.randint(2, Lt + 1, (B,), device="cuda", dtype=torch.int32)
        mask = torch.arange(Lt, device="cuda").view(1, -1) < lens.view(-1, 1)
        dec.prepare()
        for K in widths:
            tokens, parents, scores, probs, best, path = dec.beam(emb, h0, enc_a, enc_i, mask, lens, 4, K)
            assert (parents[:, :, 0] >= 0).all() and (path >= 0).all()
            sc = scores.nan_to_num(neginf=-1e38)
            assert (sc[:, :, :-1] >= sc[:, :, 1:]).all()
            assert ((best >= 0) & (best < lens.view(-1, 1))).all()
            assert torch.isfinite(probs).all()
    assert ops.BEAM_MAX_WIDTH == 8


def test_errors_are_raised_before_any_launch():
    model = _model(64)
    b = _batch(3).to("cuda")
    for w in (0, 9, -1, 2.0, True):
        with pytest.raises(ValueError, match="beam_width"):
            _summarize(model, b, 4, beam_width=w)
    with pytest.raises(ValueError, match="targets"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, beam_width=2)
    # a shape whose per-slot state does not fit beside the step's arrays: one video of 32 000 text rows at width 8
    dec = model.multimodal_att_decoder
    Lt = 32000
    enc_a, enc_i = torch.randn(1, Lt, 200, device="cuda"), torch.randn(1, Lt, 200, device="cuda")
    emb, h0 = torch.randn(1, Lt, 300, device="cuda"), torch.randn(1, 100, device="cuda")
    mask = torch.ones(1, 64, dtype=torch.bool, device="cuda")
    lens = torch.tensor([Lt], dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match="shared memory"):
        dec.beam(emb, h0, enc_a, enc_i, mask, lens, 4, 8)
    torch.cuda.synchronize()                               # nothing was launched: the device is still usable
    assert torch.equal(_summarize(model, b, 4, beam_width=2).indices, _summarize(model, b, 4, beam_width=2).indices)
