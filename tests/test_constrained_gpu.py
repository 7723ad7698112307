"""GPU: constrained summaries -- repeat blocking and a minimum summary length inside the greedy and beam roll-out kernels
(mmb_decoder_greedy_constrained_fused, mmb_decoder_beam_constrained_fused) against host loops of the fused step kernel that apply
the same rule, the constraints off against the unconstrained kernels, width 1 against greedy, constructed cases that force each
constraint to act, graph replay (Summarizer), the shapes of configs 3 and 5, and the errors."""
import math

import pytest
import torch

from mmbidaf_b200.summarize import _select
from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu

EMPTY, LIVE, DONE = 0, 1, 2
SETTINGS = [(True, 0), (False, 3), (True, 3), (True, 50)]       # (no_repeat, min_sentences); 50 is more than a transcript holds


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


def _summarize(model, b, steps, beam_width=None, no_repeat=False, min_sentences=0):
    return model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, steps, beam_width=beam_width,
                           no_repeat=no_repeat, min_sentences=min_sentences)


def _decoder_inputs(model, b):
    """What summarize hands the decoder: (emb_text, h0, enc_a, enc_i, mask, text_len int32)."""
    from mmbidaf_b200.layers.encoding import length_plan
    model.eval()
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    return b.text, h0, enc_a, enc_i, mask, length_plan(b.text_len, b.text.device).len_i32.clone()


def _eligible(mask, eos, used, kept, no_repeat, min_sentences):
    """The rule's eligibility over (..., M) given per-hypothesis used (..., M) bool and kept (...) long; eos broadcasts as kept."""
    M = mask.shape[-1]
    idx = torch.arange(M, device=mask.device)
    e = eos.unsqueeze(-1)
    avail = eos - (kept if no_repeat else 0)
    eos_ok = ((kept >= min_sentences) | (avail == 0)).unsqueeze(-1)
    below = (idx < e) & ~(used if no_repeat else torch.zeros_like(used))
    return mask & (below | ((idx == e) & eos_ok))


def _greedy_reference(dec, emb, h0, enc_a, enc_i, mask, text_len, steps, no_repeat, min_sentences):
    """The constrained greedy rule as a host loop of the fused step kernel: where(eligible, p, -1).max(1), EOS when none is."""
    from mmbidaf_b200 import ops
    with torch.no_grad():
        seq = dec._sequence(enc_a, enc_i)["seq"]
        B, Lt, H, M = seq.B, seq.Lt, seq.H, seq.M
        dev = emb.device
        mask_u8 = ops._u8(mask)
        rows = torch.arange(B, device=dev)
        eos = text_len.long() - 1
        used = torch.zeros(B, M, dtype=torch.bool, device=dev)
        kept = torch.zeros(B, dtype=torch.long, device=dev)
        sent, h = emb.new_zeros(B, emb.shape[2]), h0.reshape(B, H).contiguous()
        cell, cov = torch.zeros(B, H, device=dev), torch.zeros(B, Lt, device=dev)
        P, picks = [], []
        for _ in range(steps):
            p, h, cell, _, cov, *_ = ops.decoder_step_fwd(seq, sent.contiguous(), h, cell, cov, mask_u8)
            ok = _eligible(mask.bool(), eos, used, kept, no_repeat, min_sentences)
            val, pick = torch.where(ok, p, -1.0).max(1)
            pick = torch.where(val < 0, eos, pick)
            below = pick < eos
            kept = kept + below.long()
            used[rows[below], pick[below]] = True
            sent = emb[rows, pick.clamp(0, Lt - 1)]
            P.append(p)
            picks.append(pick)
        return torch.stack(P, 1), torch.stack(picks, 1)


def _beam_reference(dec, emb, h0, enc_a, enc_i, mask, text_len, steps, K, no_repeat, min_sentences):
    """test_beam_gpu.py's host beam loop, with every slot's used bits and kept count gathered by parent and only eligible
    sentences offered."""
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
        used = torch.zeros(B, K, M, dtype=torch.bool, device=dev)
        kept = torch.zeros(B, K, dtype=torch.long, device=dev)
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
            elig = _eligible(mask.bool().unsqueeze(1).expand(B, K, M), eos.view(B, 1).expand(B, K), used, kept, no_repeat,
                             min_sentences)
            live = (stat == LIVE).unsqueeze(2) & (p > 0) & elig
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
            below = t < eos.view(B, 1)
            used = used.gather(1, g.expand(B, K, M)) | ((sent_of == t.unsqueeze(2)) & below.unsqueeze(2))
            kept = kept.gather(1, par) + below.long()
            tok = torch.where(ok, t, -1)
            score = torch.where(ok, sc, -math.inf)
            stat = torch.where(~ok, EMPTY, torch.where(carry | (t == eos.view(B, 1)), DONE, LIVE))
        return torch.stack(T, 1), torch.stack(R, 1), torch.stack(S_, 1), torch.stack(P, 1)


def _check_summaries(rows, text_len, steps, no_repeat, min_sentences):
    """Every summary under the greedy_search rule: no duplicates with no_repeat; at least min(min_sentences, S, text_len - 1)."""
    for row, n in zip(rows, text_len):
        chosen = _select(row, int(n))
        if no_repeat:
            assert len(set(chosen)) == len(chosen), chosen
        assert len(chosen) >= min(min_sentences, steps, int(n) - 1), (chosen, int(n))


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("no_repeat,min_sentences", SETTINGS)
def test_greedy_equals_the_host_loop_of_step_kernels(tier, B, no_repeat, min_sentences):
    model = _model(64)                                     # M = 64 > Lt = 37
    b = _batch(B).to("cuda")
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    probs, picks, terms = dec.greedy(emb, h0, enc_a, enc_i, mask, 16, text_len=lens, no_repeat=no_repeat,
                                     min_sentences=min_sentences)
    rp, rpicks = _greedy_reference(dec, emb, h0, enc_a, enc_i, mask, lens, 16, no_repeat, min_sentences)
    assert terms is None
    assert torch.equal(probs, rp)
    assert torch.equal(picks, rpicks)
    _check_summaries(picks.tolist(), b.text_len, 16, no_repeat, min_sentences)


def _check_beam(model, b, steps, K, no_repeat, min_sentences):
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    tokens, parents, scores, probs, best, path = dec.beam(emb, h0, enc_a, enc_i, mask, lens, steps, K, no_repeat, min_sentences)
    rt, rp, rs, rprob = _beam_reference(dec, emb, h0, enc_a, enc_i, mask, lens, steps, K, no_repeat, min_sentences)
    assert torch.equal(tokens, rt)
    assert torch.equal(parents, rp)
    assert torch.equal(scores, rs)
    assert torch.equal(probs, rprob)
    B = tokens.shape[0]
    j = torch.zeros(B, dtype=torch.long, device=tokens.device)
    rows = torch.arange(B, device=tokens.device)
    for s in range(steps - 1, -1, -1):
        assert torch.equal(path[:, s].long(), j)
        assert torch.equal(best[:, s], tokens[rows, s, j])
        j = parents[rows, s, j].long()
    _check_summaries(best.tolist(), b.text_len, steps, no_repeat, min_sentences)


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [3, 32])
@pytest.mark.parametrize("K", [2, 4, 8])
@pytest.mark.parametrize("no_repeat,min_sentences", SETTINGS)
def test_beam_equals_the_host_loop_of_step_kernels(tier, B, K, no_repeat, min_sentences):
    _check_beam(_model(64), _batch(B).to("cuda"), 16, K, no_repeat, min_sentences)


def test_long_lecture_side_of_the_rule_equals_the_host_loops(monkeypatch):
    from mmbidaf_b200 import ops
    model = _model(700)
    b = make_batch(32, 700, 60, 6, 6, seed=41).to("cuda")
    assert ops.decoder_cut(32, 700) == "chunks"            # the constrained roll-outs run the cluster kernel; so must the references
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    _check_beam(model, b, 6, 3, True, 3)
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    probs, picks, _ = dec.greedy(emb, h0, enc_a, enc_i, mask, 6, text_len=lens, no_repeat=True, min_sentences=3)
    rp, rpicks = _greedy_reference(dec, emb, h0, enc_a, enc_i, mask, lens, 6, True, 3)
    assert torch.equal(probs, rp) and torch.equal(picks, rpicks)


@pytest.mark.parametrize("B", [1, 3, 32])
def test_constraints_off_equal_the_unconstrained_kernels(B):
    from mmbidaf_b200 import ops
    model = _model(64)
    b = _batch(B).to("cuda")
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        seq = dec._sequence(enc_a, enc_i)["seq"]
        h = h0.reshape(B, -1).contiguous()
        probs, argmax, _ = ops.decoder_greedy_fwd(seq, emb, h, ops._u8(mask), 16)
        cprobs, cpicks = ops.decoder_greedy_constrained_fwd(seq, emb, h, ops._u8(mask), lens, 16, False, 0)
        assert torch.equal(probs, cprobs) and torch.equal(argmax, cpicks)
        for K in (2, 4):
            plain = ops.decoder_beam_fwd(seq, emb, h, ops._u8(mask), lens, 16, K)
            cons = ops.decoder_beam_fwd(seq, emb, h, ops._u8(mask), lens, 16, K, constrained=True)
            assert all(torch.equal(x, y) for x, y in zip(plain, cons))


@pytest.mark.parametrize("B", [1, 3, 21])
@pytest.mark.parametrize("no_repeat,min_sentences", SETTINGS)
def test_width_one_is_the_constrained_greedy_summary(B, no_repeat, min_sentences):
    model = _model(64)
    b = _batch(B).to("cuda")
    greedy = _summarize(model, b, 16, no_repeat=no_repeat, min_sentences=min_sentences)
    beam = _summarize(model, b, 16, beam_width=1, no_repeat=no_repeat, min_sentences=min_sentences)
    assert torch.equal(beam.indices, greedy.indices) and torch.equal(beam.counts, greedy.counts)
    # distributions equal up to each video's first EOS pick, zero after (carries)
    picks = beam.beams.tokens[:, :, 0].cpu()
    for v in range(B):
        hits = (picks[v] == b.text_len[v] - 1).nonzero()
        last = int(hits[0]) if len(hits) else 15
        assert torch.equal(beam.out_distributions[v, :last + 1], greedy.out_distributions[v, :last + 1])
        assert (beam.out_distributions[v, last + 1:] == 0).all()


def test_no_repeat_blocks_a_dominant_sentence():
    model = _model(64)
    b = _batch(3).to("cuda")
    k = 2                                                  # a sentence row of videos 0 and 2 (video 1 holds one sentence)
    assert b.text_len[0] - 1 > k and b.text_len[2] - 1 > k
    with torch.no_grad():
        model.multimodal_att_decoder.out.bias[k] += 60.0
    for w in (None, 4):
        plain = _summarize(model, b, 16, beam_width=w).to_lists()
        blocked = _summarize(model, b, 16, beam_width=w, no_repeat=True).to_lists()
        for v in (0, 2):
            assert plain[v] == [k] * 16
            # (a beam may prefer a path that ends before it picks k: every pick but k costs about as much as EOS does)
            assert blocked[v].count(k) == 1 if w is None else blocked[v].count(k) <= 1
            assert len(set(blocked[v])) == len(blocked[v])


def test_min_sentences_outlasts_a_dominant_eos():
    model = _model(64)
    b = _batch(3).to("cuda")
    k = b.text_len[2] - 1                                  # video 2's EOS row
    with torch.no_grad():
        model.multimodal_att_decoder.out.bias[k] += 60.0
    for w in (None, 4):
        assert _summarize(model, b, 16, beam_width=w).to_lists()[2] == []
        got = _summarize(model, b, 16, beam_width=w, min_sentences=3).to_lists()[2]
        assert len(got) == 3, got
        got = _summarize(model, b, 16, beam_width=w, no_repeat=True, min_sentences=3).to_lists()[2]
        assert len(got) == 3 and len(set(got)) == 3, got


def test_short_transcripts():
    model = _model(64)
    b = _batch(3)
    b.text[2, 1:] = 0                                      # video 2: the EOS row alone
    b.text[2, 0] = -1.0
    b.text_len[2] = 1
    b = b.to("cuda")
    for w in (None, 1, 4):
        got = _summarize(model, b, 16, beam_width=w, no_repeat=True, min_sentences=3).to_lists()
        assert got[1] == [0]                               # one sentence and EOS: the sentence once, then EOS
        assert got[2] == []
        assert len(got[0]) >= 3 and len(set(got[0])) == len(got[0])


def test_summarizer_replays_equal_eager_constrained_summarize():
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    summarizer = Summarizer(model)
    batches = [make_batch(4, 37, 45, 7, 12, seed=s).to("cuda") for s in (1, 2, 3)]
    opts = [dict(no_repeat=True, min_sentences=3), dict(beam_width=3, no_repeat=True, min_sentences=3)]
    for o in opts:
        for b in batches:
            got = summarizer(b, **o)
            got = [t.clone() for t in got[:4] if t is not None]
            want = _summarize(model, b, b.max_dec_len, **o)
            assert all(torch.equal(g, w) for g, w in zip(got, [t for t in want[:4] if t is not None]))
    assert len(summarizer.buckets) == 2
    summarizer(batches[0], no_repeat=True)                  # another setting: a new bucket
    summarizer(batches[0])
    assert len(summarizer.buckets) == 4
    with torch.no_grad():                                   # an optimiser-style in-place update
        model.multimodal_att_decoder.out.weight.mul_(1.5)
        model.multimodal_att_decoder.W2.weight.add_(0.01)
    for o in opts:
        got = summarizer(batches[0], **o)
        want = _summarize(model, batches[0], batches[0].max_dec_len, **o)
        assert torch.equal(got.out_distributions, want.out_distributions) and torch.equal(got.indices, want.indices)


def test_constrained_roll_outs_launch_at_config3_and_config5_shapes():
    torch.manual_seed(0)
    D, H, E = 200, 100, 300
    for B, Lt, widths in ((32, 409, range(1, 9)), (16, 4096, range(1, 5))):
        model = _model(Lt)
        dec = model.multimodal_att_decoder
        model.eval()
        enc_a, enc_i = torch.randn(B, Lt, D, device="cuda"), torch.randn(B, Lt, D, device="cuda")
        emb, h0 = torch.randn(B, Lt, E, device="cuda"), torch.randn(B, 1, H, device="cuda")
        lens = torch.randint(5, Lt + 1, (B,), device="cuda", dtype=torch.int32)
        eos = lens.view(-1, 1).long() - 1
        mask = torch.arange(Lt, device="cuda").view(1, -1) < lens.view(-1, 1)
        dec.prepare()
        probs, picks, _ = dec.greedy(emb, h0, enc_a, enc_i, mask, 4, text_len=lens, no_repeat=True, min_sentences=3)
        # 4 steps under min_sentences 3: three sentences, then EOS or a fourth
        assert torch.isfinite(probs).all() and ((picks >= 0) & (picks <= eos)).all() and (picks[:, :3] < eos).all()
        for K in widths:
            tokens, parents, scores, probs, best, path = dec.beam(emb, h0, enc_a, enc_i, mask, lens, 4, K, True, 3)
            assert (parents[:, :, 0] >= 0).all() and (path >= 0).all()
            assert ((best >= 0) & (best <= eos)).all() and (best[:, :3] < eos).all()
            assert torch.isfinite(probs).all()


def test_errors_are_raised_before_any_launch():
    from mmbidaf_b200 import ops
    model = _model(64)
    b = _batch(3).to("cuda")
    before = ops.launch_count
    bad = [dict(no_repeat=1), dict(no_repeat="yes"), dict(min_sentences=-1), dict(min_sentences=2.0), dict(min_sentences=True)]
    for kw in bad:
        for w in (None, 2):
            with pytest.raises(ValueError, match="no_repeat|min_sentences"):
                _summarize(model, b, 4, beam_width=w, **kw)
    for kw in (dict(no_repeat=True), dict(min_sentences=2)):
        with pytest.raises(ValueError, match="targets"):
            model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, **kw)
    assert ops.launch_count == before
    torch.cuda.synchronize()                               # nothing was launched: the device is still usable
    got = _summarize(model, b, 4, beam_width=2, no_repeat=True, min_sentences=2)
    assert torch.equal(got.indices, _summarize(model, b, 4, beam_width=2, no_repeat=True, min_sentences=2).indices)
