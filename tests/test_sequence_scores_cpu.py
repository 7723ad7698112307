"""CPU: MMBiDAF.sequence_scores' argument checks (before any device work), the rule that folds the gradient of p_tok into the nll
coefficient, and the B200-only error."""
import math

import pytest
import torch

from mmbidaf_b200.synth import make_batch


def _model(m=64):
    from mmbidaf_b200.models import MMBiDAF
    return MMBiDAF(100, 300, 128, 1000, torch.device("cpu"), drop_prob=0.0, max_transcript_length=m)


def _call(model, b, S, cand, text=None):
    return model.sequence_scores(b.text if text is None else text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, S, cand)


def test_bad_candidates_and_text_with_grad_raise_value_error():
    model = _model()
    b = make_batch(3, 37, 45, 7, 16, seed=1)
    tok = torch.zeros(3, 2, 16, dtype=torch.int64)
    for bad in (tok[:, :, :15], tok.int(), tok[:2], torch.zeros(3, 65, 16, dtype=torch.int64), torch.zeros(3, 0, 16, dtype=torch.int64),
                tok.view(6, 16)):
        with pytest.raises(ValueError, match="sequence_scores"):
            _call(model, b, 16, bad)
    with pytest.raises(ValueError, match="candidate_tokens"):
        _call(model, b, 16, [[[0] * 17], [], []])
    with pytest.raises(ValueError, match="candidate_tokens"):
        _call(model, b, 16, [[[0]], [[0]]])
    with pytest.raises(ValueError, match="requires grad"):
        _call(model, b, 16, tok, text=b.text.clone().requires_grad_())


def test_cpu_tensors_raise_b200_only():
    model = _model()
    b = make_batch(3, 37, 45, 7, 16, seed=1)
    with pytest.raises(RuntimeError, match="B200 only"):
        _call(model, b, 16, torch.zeros(3, 2, 16, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="B200 only"):
        _call(model, b, 16, [[[0]], [[1]], [[2, 3]]])


def test_fold_rule_gives_the_p_tok_gradient():
    from mmbidaf_b200.functional import fold_step_p_grad
    g = torch.Generator().manual_seed(0)
    B, N, S = 2, 3, 4
    p = torch.rand(B, N, S, generator=g) * 0.9 + 0.05
    p[0, 1, 2] = 0.0                                               # a masked or out-of-range token
    g_terms = torch.randn(S, 2, B * N, generator=g)
    g_p = torch.randn(B, N, S, generator=g)
    g_p[0, 1, 2] = math.nan                                        # 0 * inf of log's backward: dropped
    got = fold_step_p_grad(g_terms, g_p, p)
    assert torch.equal(got[:, 1], g_terms[:, 1])
    pt, gp = p.reshape(B * N, S).t(), g_p.reshape(B * N, S).t()
    for s in range(S):
        for r in range(B * N):
            if pt[s, r] == 0:
                assert got[s, 0, r] == g_terms[s, 0, r]
                continue
            # the kernel's dp_t = -g_nll / (p + 1e-12) is the nll's share plus exactly g_p
            dp = -got[s, 0, r].double() / (pt[s, r].double() + 1e-12)
            want = -g_terms[s, 0, r].double() / (pt[s, r].double() + 1e-12) + gp[s, r].double()
            assert math.isclose(float(dp), float(want), rel_tol=1e-5, abs_tol=1e-5)
    assert torch.equal(fold_step_p_grad(None, None, p), torch.zeros(S, 2, B * N))
    assert torch.equal(fold_step_p_grad(g_terms, None, p), g_terms)
