"""GPU: sequence-level training -- the forced roll-out that saves every step (mmb_decoder_forced_train_fused) and the reverse roll-out
(mmb_decoder_forced_bwd_fused) against host loops of the step kernels, MMBiDAF.sequence_scores against the training path, the fp64
oracle, itself over candidates, score, graph replay, the launch counter and the errors."""
import copy

import pytest
import torch

from conftest import grad_err, rel_err
from oracle import mmbidaf_oracle as O
from test_sample_gpu import _batch, _decoder_inputs, _model
from test_score_gpu import _random_tokens

pytestmark = pytest.mark.gpu


@pytest.fixture
def tier(request):
    import mmbidaf_b200
    mmbidaf_b200.set_precision(request.param)
    yield request.param
    mmbidaf_b200.set_precision("fp32")


@pytest.fixture
def fused_steps(monkeypatch):
    """The host loops' step kernels are the cluster kernels at every B N (both roll-outs run them whatever decoder_cut says)."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")


def _seq(dec, enc_a, enc_i):
    with torch.no_grad():
        return dec._sequence(enc_a, enc_i)["seq"]


def _replicated(seq, N):
    """The sequence over B N rows: every video's encoder rows repeated N times (the host loops' inputs)."""
    from mmbidaf_b200 import _lib
    rs = copy.copy(seq)
    for f in ("proj_a", "proj_i", "enc_a", "enc_i"):
        setattr(rs, f, getattr(seq, f).repeat_interleave(N, 0).contiguous())
    rs.B, rs.nch = seq.B * N, _lib.lib().mmb_decoder_chunks(seq.B * N, seq.Lt)
    rs.counters = torch.zeros(2, seq.B * N, device=seq.enc_a.device, dtype=torch.int32)
    return rs


def _host_forward(seq, emb, h0, mask, tokens):
    """The forced roll-out as a host loop of mmb_decoder_step_fused_fwd over the B N replicated rows: per step (inputs, outputs)."""
    from mmbidaf_b200 import ops
    B, N, S = tokens.shape
    R, Lt, H = B * N, seq.Lt, seq.H
    rs = _replicated(seq, N)
    emb_r, mask_r = emb.repeat_interleave(N, 0), ops._u8(mask.bool().repeat_interleave(N, 0))
    rows, tok = torch.arange(R, device=emb.device), tokens.reshape(R, S)
    sent, h = emb.new_zeros(R, emb.shape[2]), h0.reshape(B, H).repeat_interleave(N, 0).contiguous()
    cell, cov = torch.zeros(R, H, device=emb.device), torch.zeros(R, Lt, device=emb.device)
    steps = []
    for s in range(S):
        t = tok[:, s].contiguous()
        out = ops.decoder_step_fwd(rs, sent.contiguous(), h, cell, cov, mask_r, target=t)
        steps.append(dict(h=h, cell=cell, cov=cov, t=t, out=out))
        probs, h, cell, _, cov, _, _, _ = out
        sent = emb_r[rows, t.clamp(0, Lt - 1)]
    return rs, steps


def _host_backward(rs, steps, g_terms, M):
    """The reverse roll-out as a host loop of mmb_decoder_step_fused_bwd, steps in reverse with d h / d cell / d cov chained.  A token
    outside 0..M-1 goes in clamped with a zero nll coefficient (the step kernel reads its p unguarded)."""
    from mmbidaf_b200 import ops
    R, D = rs.B, rs.D
    d_proj_a, d_proj_i = torch.zeros_like(rs.proj_a), torch.zeros_like(rs.proj_i)
    vec_acc, scal_acc = rs.enc_a.new_zeros(R, 6, D), rs.enc_a.new_zeros(R, 4)
    d_h = d_cell = d_cov = None
    per_step = [None] * len(steps)
    for s in reversed(range(len(steps))):
        st = steps[s]
        probs, h_out, cell_out, att, cov_out, _, saved, _ = st["out"]
        inside = (st["t"] >= 0) & (st["t"] < M)
        g = g_terms[s].clone()
        g[0] = torch.where(inside, g[0], torch.zeros_like(g[0]))
        d_h, d_cell, d_cov, d_logits, d_gates, d_ctx12, d_hw4, d_pre_b = ops.decoder_step_bwd(
            rs, st["h"], st["cell"], st["cov"], probs, cell_out, saved, None, d_h, d_cell, None, d_cov, d_proj_a, d_proj_i, vec_acc,
            scal_acc, target=st["t"].clamp(0, M - 1).contiguous(), d_lossvec=g.contiguous(), att_cov=att, cov_out=cov_out)
        per_step[s] = (d_logits, d_gates, d_hw4, d_ctx12, d_pre_b)
    return per_step, d_h, d_proj_a, d_proj_i, vec_acc, scal_acc


def _g_terms(S, R, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(S, 2, R, generator=g) * (torch.rand(S, 2, R, generator=g) > 0.25)
    return x.cuda()


def _check_kernels(dec, emb, h0, enc_a, enc_i, mask, tokens, seed=0):
    """Both kernels against the host loops: every saved slice and per-row gradient bit for bit, d_proj bit for bit at N = 1."""
    from mmbidaf_b200 import ops
    seq = _seq(dec, enc_a, enc_i)
    B, N, S = tokens.shape
    R, D, M = B * N, seq.D, seq.M
    h0r = h0.reshape(B, -1).contiguous()
    p_tok, terms, saved = ops.decoder_forced_train_fwd(seq, emb, h0r, ops._u8(mask), tokens)
    _, p_ref, t_ref = ops.decoder_forced_fwd(seq, emb, h0r, ops._u8(mask), tokens)
    assert torch.equal(p_tok, p_ref) and torch.equal(terms, t_ref)
    probs, hw, alpha, beta, ctx12, pb, xcat, gates, att_cov, cell, cov, h_last = saved
    rs, steps = _host_forward(seq, emb, h0, mask, tokens)
    assert torch.equal(cell[0], torch.zeros_like(cell[0])) and torch.equal(cov[0], torch.zeros_like(cov[0]))
    for s, st in enumerate(steps):
        p, h_out, cell_out, att, cov_out, _, sv, lv = st["out"]
        for got, want in zip((probs[s], hw[s], alpha[s], beta[s], ctx12[s], pb[s], xcat[s], gates[s], att_cov[s], cell[s + 1],
                              cov[s + 1], terms[s, 1]), (p, *sv[:2], sv[2], *sv[3:], att, cell_out, cov_out, lv[1])):
            assert torch.equal(got, want), s
        inside = (st["t"] >= 0) & (st["t"] < M)                    # (the step kernel writes no nll for a token outside 0..M-1)
        assert torch.equal(terms[s, 0][inside], lv[0][inside]), s
    assert torch.equal(h_last, steps[-1]["out"][1])
    g_terms = _g_terms(S, R, seed)
    vec_acc, scal_acc = seq.enc_a.new_zeros(R, 6, D), seq.enc_a.new_zeros(R, 4)
    d_proj_a, d_proj_i = torch.zeros_like(seq.proj_a), torch.zeros_like(seq.proj_i)
    got = ops.decoder_forced_bwd(seq, saved, tokens, g_terms, d_proj_a, d_proj_i, vec_acc, scal_acc)
    per_step, d_h0, ref_pa, ref_pi, ref_vec, ref_scal = _host_backward(rs, steps, g_terms, M)
    for s in range(S):
        for x, y in zip(got[:5], per_step[s]):
            assert torch.equal(x[s], y), s
    assert torch.equal(got[5], d_h0)
    assert torch.equal(vec_acc, ref_vec) and torch.equal(scal_acc, ref_scal)
    for x, y in ((d_proj_a, ref_pa), (d_proj_i, ref_pi)):
        y = y.view(B, N, *y.shape[1:]).sum(1)
        if N == 1:
            assert torch.equal(x, y)
        else:
            assert rel_err(x, y) <= 1e-6


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("N", [1, 4])
def test_kernels_equal_the_host_loops(tier, B, N, fused_steps):
    model = _model(64)
    b = _batch(B).to("cuda")
    emb, h0, enc_a, enc_i, mask, _ = _decoder_inputs(model, b)
    _check_kernels(model.multimodal_att_decoder, emb, h0, enc_a, enc_i, mask, _random_tokens(b.text_len, N, 12, seed=B * N), seed=B + N)


def test_kernels_with_edge_tokens_and_config3_shapes(fused_steps):
    model = _model(64)
    b = _batch(3).to("cuda")
    emb, h0, enc_a, enc_i, mask, _ = _decoder_inputs(model, b)
    tokens = _random_tokens(b.text_len, 2, 8, seed=3)
    tokens[0, 0, 2], tokens[1, 1, 0], tokens[2, 0, 5] = -3, 1 << 40, 64 + 7
    _check_kernels(model.multimodal_att_decoder, emb, h0, enc_a, enc_i, mask, tokens, seed=11)
    torch.manual_seed(0)
    D, H, E, B, Lt, S, N = 200, 100, 300, 32, 409, 12, 1
    model = _model(Lt)
    dec = model.multimodal_att_decoder
    model.eval()
    enc_a, enc_i = torch.randn(B, Lt, D, device="cuda"), torch.randn(B, Lt, D, device="cuda")
    emb, h0 = torch.randn(B, Lt, E, device="cuda"), torch.randn(B, 1, H, device="cuda")
    lens = torch.randint(5, Lt + 1, (B,), device="cuda", dtype=torch.int32)
    mask = torch.arange(Lt, device="cuda").view(1, -1) < lens.view(-1, 1)
    dec.prepare()
    _check_kernels(dec, emb, h0, enc_a, enc_i, mask, _random_tokens(lens.cpu(), N, S, seed=B), seed=5)


def _scores(model, b, S, cand):
    return model.sequence_scores(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, S, cand)


def _grads(model):
    return {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21])
def test_gradients_equal_the_training_path(tier, B):
    b = _batch(B).to("cuda")
    T = b.max_dec_len
    targets = b.targets[:, :T]
    ref = _model(64)
    ref.train()
    _, loss = ref(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, targets, b.target_len, T)
    loss.backward()
    model = _model(64)
    model.train()
    got = _scores(model, b, T, targets.reshape(B, T).long().unsqueeze(1).contiguous())
    total = got.loss[:, 0].sum()
    assert rel_err(total, loss) <= 1e-6
    total.backward()
    want, have = _grads(ref), _grads(model)
    assert set(want) == set(have)
    tol = 1e-5 if tier == "fp32" else 2e-2
    for n in want:
        assert grad_err(have[n], want[n], n) <= tol, n


def _oracle_objective(p, emb, h0, enc_a, enc_i, mask, tokens, lens, w_logp, w_loss):
    """sum over rows of w_logp logp + w_loss loss, the teacher-forced loop of the fp64 oracle's decoder step."""
    B, N, S = tokens.shape
    Lt = emb.shape[1]
    total = enc_a.new_zeros(())
    for n in range(N):
        sent = emb.new_zeros(B, 1, emb.shape[2])
        h, cell, cov = h0.reshape(B, 1, -1), h0.new_zeros(1, B, h0.shape[-1]), emb.new_zeros(B, Lt, 1)
        logp, loss = enc_a.new_zeros(B), enc_a.new_zeros(B)
        ended = torch.zeros(B, dtype=torch.bool, device=tokens.device)
        for s in range(S):
            t = tokens[:, n, s]
            probs, h, cell, att, cov = O.decoder_step(p, sent, h, cell, enc_a, enc_i, cov, mask)
            pt = probs.gather(1, t.view(-1, 1)).squeeze(1)
            loss = loss + (-torch.log(pt + 1e-12) + torch.minimum(att, cov).sum((1, 2))) / S
            logp = logp + torch.where(ended, torch.zeros_like(pt), torch.log(pt))
            ended = ended | (t == (lens - 1))
            sent = emb[torch.arange(B, device=tokens.device), t.clamp(0, Lt - 1)].unsqueeze(1)
        total = total + (w_logp[:, n] * logp).sum() + (w_loss[:, n] * loss).sum()
    return total


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("N", [1, 4])
def test_gradients_match_the_fp64_oracle(B, N):
    from mmbidaf_b200.summarize import forced_scores
    model = _model(64)
    b = _batch(B).to("cuda")
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    tokens = _random_tokens(b.text_len, N, 10, seed=B + 3 * N)
    g = torch.Generator().manual_seed(B * N)
    w_logp, w_loss = torch.randn(B, N, generator=g), torch.randn(B, N, generator=g)
    leaves = [t.detach().clone().requires_grad_() for t in (enc_a, enc_i, h0)]
    dec.zero_grad()
    p_tok, terms = dec.force_train(emb, leaves[2], leaves[0], leaves[1], mask, tokens)
    sc = forced_scores(tokens, p_tok, terms, torch.ones(B, N, dtype=torch.bool, device="cuda"), lens)
    ((sc.logp * w_logp.cuda()).sum() + (sc.loss * w_loss.cuda()).sum()).backward()
    p = {n: t.detach().double().cpu().requires_grad_() for n, t in dec.named_parameters()}
    ref_leaves = [t.detach().double().cpu().requires_grad_() for t in (enc_a, enc_i, h0)]
    obj = _oracle_objective(p, emb.double().cpu(), ref_leaves[2], ref_leaves[0], ref_leaves[1], mask.cpu(), tokens.cpu(),
                            lens.long().cpu(), w_logp.double(), w_loss.double())
    obj.backward()
    # the tolerances of the per-step path's gradient checks (tests/test_decoder_gpu.py): fp32 sums over S N rows in another order
    for n, t in dec.named_parameters():
        tol = 5e-4 if n in ("v1.bias", "v2.bias", "v_beta_1.bias", "v_beta_2.bias") else 5e-5
        assert grad_err(t.grad, p[n].grad, n) <= tol, n
    for got, want in zip(leaves, ref_leaves):
        assert grad_err(got.grad, want.grad) <= 2e-5


def test_linearity_over_candidates_and_sixty_four_candidates():
    model = _model(64)
    b = _batch(3).to("cuda")
    model.train()
    tokens = _random_tokens(b.text_len, 4, 12, seed=9)

    def grads_of(tok):
        model.zero_grad()
        sc = _scores(model, b, 12, tok)
        (sc.logp.sum() + sc.loss.sum()).backward()
        return _grads(model)
    whole = grads_of(tokens)
    parts = [grads_of(tokens[:, n:n + 1].contiguous()) for n in range(4)]
    for n in whole:
        assert grad_err(whole[n], sum(p[n] for p in parts), n) <= 1e-6, n
    # N = 64 at B = 2 (128 rows) against four calls of N = 16 (32 rows): both on 4-CTA clusters, so every row is the same
    b = _batch(2).to("cuda")
    tokens = _random_tokens(b.text_len, 64, 6, seed=1)

    def grads_of64(tok):
        model.zero_grad()
        sc = _scores(model, b, 6, tok)
        (sc.logp.sum() + sc.loss.sum()).backward()
        return _grads(model)
    whole = grads_of64(tokens)
    assert all(torch.isfinite(g).all() for g in whole.values())
    parts = [grads_of64(tokens[:, 16 * q:16 * (q + 1)].contiguous()) for q in range(4)]
    # (the weight-gradient GEMMs sum 768 rows in one call against 4 x 192: fp32 rounding at the 1e-6 level, hence 1e-5 here)
    for n in whole:
        assert grad_err(whole[n], sum(p[n] for p in parts), n) <= 1e-5, n


def test_no_grad_eval_equals_score_and_lists_path():
    model = _model(64)
    b = _batch(3).to("cuda")
    model.eval()
    tokens = _random_tokens(b.text_len, 4, 16, seed=2)
    lists = [[[0, 3, 1], [2]], [[0]], [[4, 2]]]
    for cand in (tokens, lists):
        want = model.score(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, cand)
        with torch.no_grad():
            got = _scores(model, b, 16, cand)
        for x, y in zip(got[:5], want[:5]):
            assert torch.equal(x, y)
        assert got.probs is None
    # under autograd the training roll-out: the same values, bit for bit
    got = _scores(model, b, 16, lists)
    for x, y in zip(got[:5], want[:5]):
        assert torch.equal(x.detach(), y)


def test_edge_tokens_and_invalid_rows_give_finite_and_zero_gradients():
    model = _model(64)
    b = _batch(3).to("cuda")
    model.train()
    tokens = _random_tokens(b.text_len, 2, 8, seed=4)
    tokens[0, 0, 1], tokens[1, 1, 3], tokens[2, 0, 0] = -1, 64, 63       # below 0, M, and a row hidden by the mask
    model.zero_grad()
    sc = _scores(model, b, 8, tokens)
    (sc.step_p.sum() + sc.loss.sum()).backward()
    assert all(torch.isfinite(g).all() for g in _grads(model).values())
    # video 2 holds no candidate (invalid rows only): its rows add nothing
    model.zero_grad()
    sc = _scores(model, b, 8, [[[0, 3]], [[0]], []])
    assert sc.valid.tolist() == [[True], [True], [False]]
    torch.where(sc.valid, sc.logp, torch.zeros_like(sc.logp)).sum().backward()
    with_invalid = _grads(model)
    model.zero_grad()
    sc = _scores(model, b, 8, [[[0, 3]], [[0]], [[1]]])
    (sc.logp * torch.tensor([[1.0], [1.0], [0.0]], device="cuda")).sum().backward()
    for n, g in _grads(model).items():
        assert rel_err(with_invalid[n], g) <= 1e-6, n


def _captured(fn):
    """fn() eagerly, then captured into a CUDA graph and replayed once: (eager results, replayed results)."""
    eager = [g.clone() for g in fn()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    graph.replay()
    torch.cuda.synchronize()
    return eager, out


def test_graph_capture_equals_eager_and_two_launches():
    from mmbidaf_b200 import ops
    ops.rng_next_keys("cuda", 1)
    for N in (1, 3):
        model = _model(64)
        b = _batch(3).to("cuda")
        tokens = _random_tokens(b.text_len, N, 10, seed=N)
        dec = model.multimodal_att_decoder
        emb, h0, enc_a, enc_i, mask, _ = _decoder_inputs(model, b)
        leaves = [t.detach().clone().requires_grad_() for t in (enc_a, enc_i, h0)]
        dparams = list(dec.parameters())

        def decoder_part():                                     # the forced roll-out and its backward on fixed encoder outputs
            for t in leaves + dparams:
                t.grad = None
            p_tok, terms = dec.force_train(emb, leaves[2], leaves[0], leaves[1], mask, tokens)
            (p_tok.sum() + terms.sum()).backward()
            return [t.grad for t in leaves + dparams]
        eager, out = _captured(decoder_part)
        names = ["enc_a", "enc_i", "h0"] + [n for n, _ in dec.named_parameters()]
        bad = [(n, float((g - e).abs().max()), float(e.abs().max())) for n, g, e in zip(names, out, eager)
               if not (torch.equal(g, e) if N == 1 else grad_err(g, e, n) <= 1e-6)]
        assert not bad, (N, bad)
        params = list(model.parameters())
        model.train()

        def whole():                                            # sequence_scores + backward: no host sync, capturable
            for p in params:
                p.grad = None
            sc = _scores(model, b, 10, tokens)
            (sc.logp.sum() + sc.loss.sum()).backward()
            return [p.grad for p in params if p.grad is not None]
        eager, out = _captured(whole)
        assert len(out) == len(eager)
        names = [n for n, p in model.named_parameters() if p.grad is not None]
        bad = [(n, float((g - e).abs().max()), float(e.abs().max())) for n, g, e in zip(names, out, eager)
               if not (torch.equal(g, e) if N == 1 else grad_err(g, e, n) <= 1e-6)]
        assert not bad, (N, bad)
    # the decoder part is two library kernels whatever S is
    model = _model(64)
    b = _batch(3).to("cuda")
    dec = model.multimodal_att_decoder
    emb, h0, enc_a, enc_i, mask, _ = _decoder_inputs(model, b)
    for S in (3, 14):
        leaves = [t.detach().clone().requires_grad_() for t in (enc_a, enc_i)]
        tok = _random_tokens(b.text_len, 2, S, seed=S)
        before = ops.launch_count
        p_tok, terms = dec.force_train(emb, h0, leaves[0], leaves[1], mask, tok)
        mid = ops.launch_count
        (p_tok.sum() + terms.sum()).backward()
        # forward: the two hoisted projections' products are torch GEMMs; the kernels counted are the roll-out's
        assert mid - before == 1
        assert ops.launch_count - mid == 1 + 2 * 2                             # the reverse roll-out + two bias col_sums
    torch.cuda.synchronize()


def test_errors():
    from mmbidaf_b200 import _lib, ops
    model = _model(64)
    b = _batch(3).to("cuda")
    model.train()
    tok = torch.zeros(3, 2, 16, dtype=torch.int64, device="cuda")
    before = ops.launch_count
    for bad in (tok[:, :, :15], tok.int(), tok[:2], torch.zeros(3, 65, 16, dtype=torch.int64, device="cuda"), tok.cpu(),
                torch.zeros(3, 0, 16, dtype=torch.int64, device="cuda")):
        with pytest.raises(ValueError, match="sequence_scores"):
            _scores(model, b, 16, bad)
    with pytest.raises(ValueError, match="candidate_tokens"):
        _scores(model, b, 16, [[[0] * 17], [], []])
    with pytest.raises(ValueError, match="requires grad"):
        model.sequence_scores(b.text.clone().requires_grad_(), b.text_len, b.audio, b.audio_len, b.images, b.image_len, 16, tok)
    assert ops.launch_count == before
    sc = _scores(model, b, 16, tok)
    total = sc.loss.sum()
    total.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="twice"):
        total.backward()
    L = _lib.lib()
    x = torch.zeros(64, device="cuda")
    t = torch.zeros(64, dtype=torch.int64, device="cuda")

    def fwd(B=1, Lt=4, D=8, M=4, S=2, N=2, tokens=t.data_ptr(), probs=x.data_ptr()):
        args = [x.data_ptr()] * 24 + [tokens, probs] + [x.data_ptr()] * 13
        return L.mmb_decoder_forced_train_fused(*args, B, Lt, D, 4, 4, M, S, N, _lib.stream())

    def bwd(B=1, Lt=4, D=8, M=4, S=2, N=2, tokens=t.data_ptr(), g=x.data_ptr()):
        args = [x.data_ptr(), tokens, g] + [x.data_ptr()] * 24 + [8, x.data_ptr(), 4096] + [x.data_ptr()] * 7
        return L.mmb_decoder_forced_bwd_fused(*args, B, Lt, D, 4, M, S, N, _lib.stream())
    for call in (fwd, bwd):
        for kw in (dict(N=0), dict(N=65), dict(S=0), dict(S=-1), dict(tokens=None), dict(B=0)):
            assert call(**kw) == 1, (call, kw)                          # MMB_ERR_INVALID
        assert call(D=300) == 2                                        # MMB_ERR_UNSUPPORTED: D > 256
        assert call(Lt=1 << 20) == 2                                   # MMB_ERR_UNSUPPORTED: shared memory
    assert fwd(probs=None) == 1 and bwd(g=None) == 1
    torch.cuda.synchronize()                                           # nothing was launched: the device is still usable
