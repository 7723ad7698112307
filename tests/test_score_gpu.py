"""GPU: summary scoring -- the teacher-forced roll-out of given token rows as one cluster kernel (mmb_decoder_forced_fused) against a
host loop of the fused step kernel, against the sampled, greedy and beam roll-outs that chose the rows, against the fp64 oracle and
the training forward, the lists path, graph replay, the shapes of configs 3 and 5, and the errors."""
import copy
import math

import pytest
import torch

from conftest import rel_err
from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O
from test_sample_gpu import _batch, _decoder_inputs, _model, _summarize

pytestmark = pytest.mark.gpu


@pytest.fixture
def tier(request):
    import mmbidaf_b200
    mmbidaf_b200.set_precision(request.param)
    yield request.param
    mmbidaf_b200.set_precision("fp32")


@pytest.fixture
def fused_steps(monkeypatch):
    """The host loop's step kernel is the cluster kernel at every B N (the forced roll-out runs it whatever decoder_cut says)."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")


def _forced_reference(dec, emb, h0, enc_a, enc_i, mask, tokens):
    """The rule as a host loop over B N rows: the fused step kernel on the B-video tensors replicated row-wise, each row's token as
    the step kernel's target, the clamped row of the text as the next input."""
    from mmbidaf_b200 import _lib, ops
    with torch.no_grad():
        seq = dec._sequence(enc_a, enc_i)["seq"]
        B, N, S = tokens.shape
        Lt, H, M = seq.Lt, seq.H, seq.M
        R, dev = B * N, emb.device
        rs = copy.copy(seq)
        for f in ("proj_a", "proj_i", "enc_a", "enc_i"):
            setattr(rs, f, getattr(seq, f).repeat_interleave(N, 0).contiguous())
        rs.B, rs.nch = R, _lib.lib().mmb_decoder_chunks(R, Lt)
        rs.counters = torch.zeros(2, R, device=dev, dtype=torch.int32)
        emb_r, mask_r = emb.repeat_interleave(N, 0), ops._u8(mask.bool().repeat_interleave(N, 0))
        rows = torch.arange(R, device=dev)
        tok = tokens.reshape(R, S)
        sent, h = emb.new_zeros(R, emb.shape[2]), h0.reshape(B, H).repeat_interleave(N, 0).contiguous()
        cell, cov = torch.zeros(R, H, device=dev), torch.zeros(R, Lt, device=dev)
        P, T = [], []
        for s in range(S):
            t = tok[:, s].contiguous()
            p, h, cell, _, cov, _, _, lv = ops.decoder_step_fwd(rs, sent.contiguous(), h, cell, cov, mask_r, target=t)
            sent = emb_r[rows, t.clamp(0, Lt - 1)]
            P.append(p)
            T.append(lv)
        probs = torch.stack(P, 1).view(B, N, S, M)
        return probs, probs.gather(3, tokens.unsqueeze(3)).squeeze(3), torch.stack(T)


def _check_host_loop(dec, emb, h0, enc_a, enc_i, mask, tokens):
    probs, p_tok, terms = dec.force(emb, h0, enc_a, enc_i, mask, tokens, want_probs=True)
    rp, rt, rterms = _forced_reference(dec, emb, h0, enc_a, enc_i, mask, tokens)
    assert torch.equal(probs, rp)
    assert torch.equal(p_tok, rt)
    assert torch.equal(terms, rterms)
    _, p_tok2, terms2 = dec.force(emb, h0, enc_a, enc_i, mask, tokens)      # without the rows: the same scores
    assert torch.equal(p_tok2, p_tok) and torch.equal(terms2, terms)


def _random_tokens(lens, N, S, seed):
    """(B, N, S) int64 on the device: each video's tokens in 0..text_len-1 (EOS included, so some rows end early)."""
    g = torch.Generator().manual_seed(seed)
    lens = [int(x) for x in lens]
    return torch.stack([torch.randint(0, n, (N, S), generator=g) for n in lens]).cuda()


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("N", [1, 4])
def test_forced_equals_the_host_loop(tier, B, N, fused_steps):
    model = _model(64)
    b = _batch(B).to("cuda")
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    _check_host_loop(model.multimodal_att_decoder, emb, h0, enc_a, enc_i, mask, _random_tokens(b.text_len, N, 16, seed=B * N))


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("N", [1, 4])
def test_scores_reproduce_the_samples(tier, B, N):
    model = _model(64)
    b = _batch(B).to("cuda")
    smp = _summarize(model, b, 16, num_samples=N, temperature=1.5, seed=B + N).samples
    got = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, smp.tokens, probs=True)
    assert torch.equal(got.tokens, smp.tokens)
    assert torch.equal(got.probs, smp.probs)
    assert torch.equal(got.step_p, smp.probs.gather(3, smp.tokens.unsqueeze(3)).squeeze(3))
    assert torch.equal(got.logp, smp.logp)
    assert got.valid.all() and torch.isfinite(got.loss).all()


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
def test_scores_reproduce_the_greedy_roll_out(tier, B):
    from mmbidaf_b200 import ops
    from mmbidaf_b200.summarize import path_logp
    model = _model(64)
    b = _batch(B).to("cuda")
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    assert ops.decoder_cut(B, emb.shape[1]) == "fused"
    gprobs, argmax, _ = dec.greedy(emb, h0, enc_a, enc_i, mask, 16)
    probs, p_tok, _ = dec.force(emb, h0, enc_a, enc_i, mask, argmax.unsqueeze(1), want_probs=True)
    assert torch.equal(probs[:, 0], gprobs)
    # the greedy summary as a host list: its logp up to its first EOS
    summary = _summarize(model, b, 16)
    got = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, [[x] for x in summary.to_lists()])
    want = path_logp(gprobs.gather(2, argmax.unsqueeze(2)).squeeze(2).unsqueeze(1), argmax.unsqueeze(1), lens)
    assert torch.equal(got.logp, want)
    assert got.valid.all()


@pytest.mark.parametrize("B", [1, 3, 21])
@pytest.mark.parametrize("K", [2, 4])
def test_scores_of_the_beam_paths(B, K):
    model = _model(64)
    b = _batch(B).to("cuda")
    beams = _summarize(model, b, 16, beam_width=K).beams
    hyps = beams.paths()
    n = max(len(h) for h in hyps)
    rows = [[h[min(j, len(h) - 1)][0] for j in range(n)] for h in hyps]
    tokens = torch.tensor(rows, dtype=torch.int64, device="cuda")
    got = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, tokens)
    for v, h in enumerate(hyps):
        for j, (_, score) in enumerate(h):
            # a different cluster size (B videos against B n rows) sums the mat-vecs in another order: fp32 rounding, not bit for bit
            assert math.isclose(float(got.logp[v, j]), score, rel_tol=1e-5, abs_tol=1e-4), (v, j, float(got.logp[v, j]), score)


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("N", [1, 4])
def test_scores_match_the_fp64_oracle(tier, B, N):
    m = 64
    params = O.make_params(100, 300, 128, 1000, m, seed=224)
    model = _model(m)
    cpu = _batch(B)
    b = cpu.to("cuda")
    tokens = _random_tokens(cpu.text_len, N, 16, seed=7 * B + N)
    got = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, tokens, probs=True)
    tol = 1e-5 if tier == "fp32" else 2e-2
    for n in range(N):
        with torch.no_grad():
            want, want_loss = O.mmbidaf_forward(params, cpu.text, cpu.text_len, cpu.audio, cpu.audio_len, cpu.images.flatten(2),
                                                cpu.image_len, tokens[:, n].cpu(), 16, m, training=True, fast_lstm=True)
        assert rel_err(got.probs[:, n], want) <= tol
        assert rel_err(got.loss[:, n].sum(), want_loss) <= tol


@pytest.mark.parametrize("B", [1, 3, 21])
def test_training_forward_loss_is_the_sum_of_the_row_losses(B):
    model = _model(64)
    b = _batch(B).to("cuda")
    T = b.max_dec_len
    targets = b.targets[:, :T]
    model.train()
    with torch.no_grad():
        out, loss = model(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, targets, b.target_len, T)
    tokens = targets.reshape(B, T).long().unsqueeze(1).contiguous()
    got = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, T, tokens, probs=True)
    assert model.training                                          # the caller's flag is given back
    assert rel_err(got.loss.sum(), loss) < 1e-5
    assert rel_err(got.probs[:, 0], out) < 1e-5


def test_lists_path_and_out_of_range_tokens(fused_steps):
    model = _model(64)
    b = _batch(3).to("cuda")
    lens = [int(x) for x in b.text_len]
    assert lens[1] == 2                                            # the two-row transcript: one sentence and the EOS row
    got = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16,
                      [[[0, 3, 1], [2]], [[0]], []])
    assert got.tokens.shape == (3, 2, 16)
    assert got.valid.tolist() == [[True, True], [True, False], [False, False]]
    assert got.logp[1, 1] == -math.inf and got.loss[1, 1] == math.inf and (got.logp[2] == -math.inf).all()
    assert (got.loss[2] == math.inf).all()
    assert torch.isfinite(got.logp[0]).all() and torch.isfinite(got.loss[0]).all() and torch.isfinite(got.logp[1, 0])
    assert got.tokens[1, 0].tolist() == [0] + [1] * 15
    with pytest.raises(ValueError, match="candidate_tokens"):
        model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, [[[1]], [[1]], [[0]]])   # 1 is EOS of video 1
    # out-of-range tensor tokens: p 0, nll -log(1e-12), and the next input is the clamped row
    emb, h0, enc_a, enc_i, mask, _ = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    Lt, M = emb.shape[1], 64
    tokens = _random_tokens(b.text_len, 2, 8, seed=3)
    bad = tokens.clone()
    bad[0, 0, 2], bad[1, 1, 0], bad[2, 0, 5] = -3, 1 << 40, M + 7
    probs, p_tok, terms = dec.force(emb, h0, enc_a, enc_i, mask, bad, want_probs=True)
    clamped = bad.clamp(0, Lt - 1)
    cprobs, _, cterms = dec.force(emb, h0, enc_a, enc_i, mask, clamped, want_probs=True)
    assert torch.equal(probs, cprobs)                              # the distributions follow the clamped rows
    nll_floor = -torch.log(torch.tensor(1e-12, device="cuda"))
    for v, n, s in ((0, 0, 2), (1, 1, 0), (2, 0, 5)):
        assert p_tok[v, n, s] == 0
        assert torch.allclose(terms[s, 0, v * 2 + n], nll_floor, rtol=1e-6, atol=0)
    assert torch.equal(terms[:, 1], cterms[:, 1])                  # the coverage terms do not depend on the token's p
    rows_ok = bad == clamped
    assert torch.equal(p_tok[rows_ok], probs.gather(3, clamped.unsqueeze(3)).squeeze(3)[rows_ok])


def test_summarizer_score_replays_eager_and_sees_weight_updates():
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    b1 = make_batch(4, 37, 45, 7, 12, seed=3).to("cuda")
    b2 = make_batch(4, 37, 45, 7, 12, seed=4).to("cuda")
    t1 = _summarize(model, b1, 12, num_samples=3, seed=1).samples.tokens
    t2 = _summarize(model, b2, 12, num_samples=3, seed=2).samples.tokens
    summarizer = Summarizer(model)

    def eager(b, t):
        return model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 12, t, probs=True)

    def same(x, y):
        assert all(torch.equal(u, w) for u, w in zip(x, y))

    same(summarizer.score(b1, t1, probs=True), eager(b1, t1))
    same(summarizer.score(b2, t2, probs=True), eager(b2, t2))
    same(summarizer.score(b1, t1, probs=True), eager(b1, t1))
    assert len(summarizer.score_buckets) == 1 and len(summarizer.buckets) == 0
    before = summarizer.score(b1, t1, probs=True).logp.clone()
    with torch.no_grad():
        model.multimodal_att_decoder.out.bias.add_(torch.linspace(-0.5, 0.5, 64, device="cuda"))
    after = summarizer.score(b1, t1, probs=True)
    assert not torch.equal(after.logp, before)
    same(after, eager(b1, t1))
    with pytest.raises(ValueError, match="Summarizer.score"):
        summarizer.score(b1, t1.int())


def test_forced_roll_outs_at_config3_and_config5_shapes(fused_steps):
    torch.manual_seed(0)
    D, H, E = 200, 100, 300
    for B, Lt, S, N in ((32, 409, 12, 8), (16, 4096, 16, 4)):
        model = _model(Lt)
        dec = model.multimodal_att_decoder
        model.eval()
        enc_a, enc_i = torch.randn(B, Lt, D, device="cuda"), torch.randn(B, Lt, D, device="cuda")
        emb, h0 = torch.randn(B, Lt, E, device="cuda"), torch.randn(B, 1, H, device="cuda")
        lens = torch.randint(5, Lt + 1, (B,), device="cuda", dtype=torch.int32)
        mask = torch.arange(Lt, device="cuda").view(1, -1) < lens.view(-1, 1)
        dec.prepare()
        _check_host_loop(dec, emb, h0, enc_a, enc_i, mask, _random_tokens(lens.cpu(), N, S, seed=B))


def test_errors_and_the_exported_symbol():
    from mmbidaf_b200 import _lib, ops
    model = _model(64)
    b = _batch(3).to("cuda")
    before = ops.launch_count
    tok = torch.zeros(3, 2, 16, dtype=torch.int64, device="cuda")
    for bad in (tok[:, :, :15], tok.int(), tok[:2], torch.zeros(3, 65, 16, dtype=torch.int64, device="cuda"), tok.cpu(),
                torch.zeros(3, 0, 16, dtype=torch.int64, device="cuda")):
        with pytest.raises(ValueError, match="score"):
            model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, bad)
    with pytest.raises(ValueError, match="candidate_tokens"):
        model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, [[[0] * 17], [], []])
    with pytest.raises(ValueError, match="score"):
        model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, tok, probs=1)
    assert ops.launch_count == before
    L = _lib.lib()
    assert hasattr(L, "mmb_decoder_forced_fused")
    x = torch.zeros(64, device="cuda")
    t = torch.zeros(64, dtype=torch.int64, device="cuda")

    def call(B=1, Lt=4, D=8, M=4, S=2, N=2, tokens=t.data_ptr(), p_tok=x.data_ptr(), terms=x.data_ptr()):
        args = [x.data_ptr()] * 24 + [tokens, None, p_tok, terms]
        return L.mmb_decoder_forced_fused(*args, B, Lt, D, 4, 4, M, S, N, _lib.stream())
    for kw in (dict(N=0), dict(N=65), dict(S=0), dict(S=-1), dict(tokens=None), dict(p_tok=None), dict(terms=None), dict(B=0)):
        assert call(**kw) == 1, kw                                 # MMB_ERR_INVALID
    assert call(D=300) == 2                                        # MMB_ERR_UNSUPPORTED: D > 256
    assert call(Lt=1 << 20) == 2                                   # MMB_ERR_UNSUPPORTED: the step's arrays exceed shared memory
    torch.cuda.synchronize()                                       # nothing was launched: the device is still usable
    got = _summarize(model, b, 4, num_samples=2, seed=1)
    assert got.samples.tokens.shape == (3, 2, 4)
