"""GPU parity: fused BiDAF kernels (through the C ABI) vs the oracle and the reference's golden vectors."""
import pytest
import torch

from conftest import grad_err, load_golden, rel_err
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu
FP32_TOL = 1e-5       # north_star: rel <= 1e-5 on the fp32 path


def _run(g_state, text, modality, tmask, mmask, keep_c=None, keep_q=None, p=0.0, precision=0):
    from mmbidaf_b200 import ops
    dev = "cuda"
    cu = lambda t: None if t is None else t.to(dev)
    out, q2c, lse_r, lse_c = ops.bidaf_fwd(cu(text), cu(modality), cu(tmask), cu(mmask), cu(g_state["text_weight"]),
                                           cu(g_state["modality_weight"]), cu(g_state["text_modality_weight"]),
                                           cu(g_state["bias"]), cu(keep_c), cu(keep_q), 1.0 / (1.0 - p), precision)
    torch.cuda.synchronize()
    return out.cpu(), q2c.cpu(), lse_r.cpu(), lse_c.cpu()


@pytest.mark.parametrize("name", ["bidaf_small.pt", "bidaf_d200.pt"])
def test_forward_matches_reference_golden(name):
    g = load_golden(name)
    out, q2c, lse_r, lse_c = _run(g["state"], g["text"], g["modality"], g["text_mask"], g["modality_mask"])
    assert rel_err(out, g["out"]) < FP32_TOL
    # saved statistics against the reference's own similarity matrix
    s = g["similarity"]
    neg = torch.full_like(s, -1e30)
    lse_row = torch.logsumexp(torch.where(g["modality_mask"].unsqueeze(1), s, neg), dim=2)
    lse_col = torch.logsumexp(torch.where(g["text_mask"].unsqueeze(2), s, neg), dim=1)
    assert rel_err(lse_r, lse_row) < FP32_TOL and rel_err(lse_c, lse_col) < FP32_TOL
    # exact structure of the output: block 0 is the text itself, bit for bit
    d = g["text"].shape[2]
    assert torch.equal(out[:, :, :d], g["text"])


@pytest.mark.parametrize("name", ["bidaf_small.pt", "bidaf_d200.pt"])
def test_forward_training_dropout_matches_reference_golden(name):
    import torch.nn.functional as F
    g = load_golden(name)
    pr = g["train_drop_prob"]
    torch.manual_seed(g["train_seed"])
    keep_c = F.dropout(torch.ones_like(g["text"]), pr, True) != 0
    keep_q = F.dropout(torch.ones_like(g["modality"]), pr, True) != 0
    out, *_ = _run(g["state"], g["text"], g["modality"], g["text_mask"], g["modality_mask"], keep_c, keep_q, pr)
    assert rel_err(out, g["train_out"]) < FP32_TOL


@pytest.mark.parametrize("shape", [(1, 1, 1, 4), (2, 5, 3, 8), (3, 64, 32, 200), (2, 65, 33, 200), (2, 130, 257, 200),
                                   (4, 100, 70, 64), (2, 40, 50, 256), (2, 31, 95, 12)])
def test_forward_matches_oracle_ragged(shape):
    bsz, lc, lq, d = shape
    gen = torch.Generator().manual_seed(1000 + lc * 7 + lq)
    p = {"text_weight": torch.randn(d, 1, generator=gen) * 0.2, "modality_weight": torch.randn(d, 1, generator=gen) * 0.2,
         "text_modality_weight": torch.randn(1, 1, d, generator=gen) * 0.2, "bias": torch.tensor([0.3])}
    text = torch.randn(bsz, lc, d, generator=gen)
    modality = torch.randn(bsz, lq, d, generator=gen)
    c_len = torch.randint(1, lc + 1, (bsz,), generator=gen).tolist()
    q_len = torch.randint(1, lq + 1, (bsz,), generator=gen).tolist()
    c_len[0], q_len[0] = lc, lq
    tmask, mmask = O.length_mask(lc, c_len), O.length_mask(lq, q_len)
    want = O.bidaf_attention({k: v.double() for k, v in p.items()}, text.double(), modality.double(), tmask, mmask)  # fp64 oracle
    out, q2c, *_ = _run(p, text, modality, tmask, mmask)
    assert rel_err(out, want) < FP32_TOL
    # exact zeros in blocks 0, 2, 3 of rows whose text is zero padding
    text_z = text.clone()
    for b, n in enumerate(c_len):
        text_z[b, n:] = 0
    out_z, *_ = _run(p, text_z, modality, tmask, mmask)
    for b, n in enumerate(c_len):
        if n < lc:
            assert (out_z[b, n:, :d] == 0).all() and (out_z[b, n:, 2 * d:] == 0).all()
            assert out_z[b, n:, d:2 * d].abs().max() > 0


def test_fully_masked_softmax_is_uniform_like_reference():
    """attention.py:94 uses -1e30, not -inf: an all-masked soft-max is uniform, not NaN."""
    gen = torch.Generator().manual_seed(5)
    d, lc, lq = 8, 6, 5
    p = {"text_weight": torch.randn(d, 1, generator=gen), "modality_weight": torch.randn(d, 1, generator=gen),
         "text_modality_weight": torch.randn(1, 1, d, generator=gen), "bias": torch.tensor([0.0])}
    text, modality = torch.randn(2, lc, d, generator=gen), torch.randn(2, lq, d, generator=gen)
    tmask = O.length_mask(lc, [6, 0])
    mmask = O.length_mask(lq, [0, 5])
    want = O.bidaf_attention(p, text, modality, tmask, mmask)
    out, *_ = _run(p, text, modality, tmask, mmask)
    assert torch.isfinite(out).all() and rel_err(out, want) < FP32_TOL


def test_unsupported_shape_raises():
    from mmbidaf_b200 import ops
    t = torch.randn(1, 4, 6, device="cuda")
    m = torch.ones(1, 4, dtype=torch.bool, device="cuda")
    w = torch.randn(6, device="cuda")
    with pytest.raises(RuntimeError, match="d=6"):
        ops.bidaf_fwd(t, t, m, m, w, w, w, torch.zeros(1, device="cuda"))


# ------------------------------------------------------------------------------------------------------------
# Tensor-core tier (tcgen05 + TMEM + TMA, bf16 operands): north_star tolerance rel <= 2e-2
# ------------------------------------------------------------------------------------------------------------
BF16_TOL = 2e-2


@pytest.mark.parametrize("name", ["bidaf_small.pt", "bidaf_d200.pt"])
def test_bf16_tier_matches_reference_golden(name):
    g = load_golden(name)
    out, q2c, lse_r, lse_c = _run(g["state"], g["text"], g["modality"], g["text_mask"], g["modality_mask"], precision=1)
    assert rel_err(out, g["out"]) < BF16_TOL
    d = g["text"].shape[2]
    assert torch.equal(out[:, :, :d], g["text"])               # block 0 stays the exact fp32 text
    s = g["similarity"]
    neg = torch.full_like(s, -1e30)
    lse_row = torch.logsumexp(torch.where(g["modality_mask"].unsqueeze(1), s, neg), dim=2)
    assert rel_err(lse_r, lse_row) < BF16_TOL


@pytest.mark.parametrize("name", ["bidaf_small.pt", "bidaf_d200.pt"])
def test_bf16_tier_training_dropout_matches_reference_golden(name):
    import torch.nn.functional as F
    g = load_golden(name)
    pr = g["train_drop_prob"]
    torch.manual_seed(g["train_seed"])
    keep_c = F.dropout(torch.ones_like(g["text"]), pr, True) != 0
    keep_q = F.dropout(torch.ones_like(g["modality"]), pr, True) != 0
    out, *_ = _run(g["state"], g["text"], g["modality"], g["text_mask"], g["modality_mask"], keep_c, keep_q, pr, precision=1)
    assert rel_err(out, g["train_out"]) < BF16_TOL


@pytest.mark.parametrize("shape", [(1, 1, 1, 8), (2, 5, 3, 8), (3, 64, 128, 200), (2, 65, 129, 200), (2, 130, 257, 200),
                                   (4, 100, 70, 64), (2, 300, 520, 200), (3, 409, 1024, 200)])
def test_bf16_tier_matches_oracle_ragged(shape):
    bsz, lc, lq, d = shape
    gen = torch.Generator().manual_seed(2000 + lc * 7 + lq)
    p = {"text_weight": torch.randn(d, 1, generator=gen) * 0.1, "modality_weight": torch.randn(d, 1, generator=gen) * 0.1,
         "text_modality_weight": torch.randn(1, 1, d, generator=gen) * 0.1, "bias": torch.tensor([0.3])}
    text = torch.randn(bsz, lc, d, generator=gen)
    modality = torch.randn(bsz, lq, d, generator=gen)
    c_len = torch.randint(1, lc + 1, (bsz,), generator=gen).tolist()
    q_len = torch.randint(1, lq + 1, (bsz,), generator=gen).tolist()
    c_len[0], q_len[0] = lc, lq
    tmask, mmask = O.length_mask(lc, c_len), O.length_mask(lq, q_len)
    want = O.bidaf_attention({k: v.double() for k, v in p.items()}, text.double(), modality.double(), tmask, mmask)
    out, q2c, lse_r, lse_c = _run(p, text, modality, tmask, mmask, precision=1)
    assert torch.isfinite(out).all()
    assert rel_err(out, want) < BF16_TOL
    fp32_out, fp32_q2c, *_ = _run(p, text, modality, tmask, mmask, precision=0)
    assert rel_err(q2c, fp32_q2c) < BF16_TOL


def test_bf16_tier_fully_masked_is_uniform_and_large_logits_are_stable():
    gen = torch.Generator().manual_seed(6)
    d, lc, lq = 8, 70, 130
    p = {"text_weight": torch.randn(d, 1, generator=gen), "modality_weight": torch.randn(d, 1, generator=gen),
         "text_modality_weight": torch.randn(1, 1, d, generator=gen) * 3, "bias": torch.tensor([0.0])}
    text, modality = torch.randn(2, lc, d, generator=gen) * 3, torch.randn(2, lq, d, generator=gen) * 3   # logits ~ +-100
    tmask = O.length_mask(lc, [lc, 0])
    mmask = O.length_mask(lq, [0, lq])
    want = O.bidaf_attention({k: v.double() for k, v in p.items()}, text.double(), modality.double(), tmask, mmask)
    out, *_ = _run(p, text, modality, tmask, mmask, precision=1)
    assert torch.isfinite(out).all() and rel_err(out, want) < 5e-2      # bf16 logits of magnitude 100: looser


# ------------------------------------------------------------------------------------------------------------
# Backward: the reference gets it from autograd (loss.backward(), train.py:148); here it is a fused kernel chain
# (csrc/bidaf_bwd_tc.cu) on the bf16 tier and the closed form on fp32 library GEMMs on the fp32 tier.
# ------------------------------------------------------------------------------------------------------------
BWD_TOL = {0: 2e-4, 1: 5e-2}      # max|d| / max|ref| per gradient tensor


def _grads(state, text, modality, tmask, mmask, grad_out, keep_c=None, keep_q=None, p=0.0, precision=0):
    from mmbidaf_b200 import functional as F
    cu = lambda t: None if t is None else t.cuda()
    c, q = text.cuda().requires_grad_(True), modality.cuda().requires_grad_(True)
    w = {k: v.cuda().requires_grad_(True) for k, v in state.items()}
    out = F.bidaf_attention(c, q, cu(tmask), cu(mmask), w["text_weight"], w["modality_weight"], w["text_modality_weight"],
                            w["bias"], cu(keep_c), cu(keep_q), 1.0 / (1.0 - p), precision)
    out.backward(grad_out.cuda())
    torch.cuda.synchronize()
    return c.grad.cpu(), q.grad.cpu(), {k: v.grad.cpu() for k, v in w.items()}


def _ds_abs_sum(state, text, modality, tmask, mmask, grad_out, keep_c=None, keep_q=None, p=0.0):
    """sum |dS| of the fp64 oracle: the scale of the (identically zero) bias gradient's rounding noise."""
    pd = {k: v.double() for k, v in state.items()}
    c, q = text.double(), modality.double()
    s = O.bidaf_similarity(pd, c, q, keep_c, keep_q, p).requires_grad_(True)
    s1 = O.masked_softmax(s, mmask.unsqueeze(1), dim=2)
    s2 = O.masked_softmax(s, tmask.unsqueeze(2), dim=1)
    a = torch.bmm(s1, q)
    b = torch.bmm(torch.bmm(s1, s2.transpose(1, 2)), c)
    torch.cat([c, a, c * a, c * b], dim=2).backward(grad_out.double())
    return float(s.grad.abs().sum())


def _check_grads(got, want_c, want_q, want_w, tol, ds_scale=None, w_floor=1e-3, bias_slack=0.0):
    dc, dq, dw = got
    errs = {"d_text": grad_err(dc, want_c), "d_modality": grad_err(dq, want_q)}
    for k, v in want_w.items():
        if k == "bias" and ds_scale is not None:
            # d loss / d bias = sum(dS) = 0 identically (both soft-maxes are shift invariant); what any implementation
            # returns is rounding noise, which for bf16 operands scales with sum |dS| (observed <= 3e-4 of it)
            errs[k] = float(dw[k].abs().max()) / (2e-3 * ds_scale + bias_slack + 1e-30) * tol
        else:
            errs[k] = grad_err(dw[k], v, k, floor=w_floor)
    assert all(e < tol for e in errs.values()), errs


@pytest.mark.parametrize("precision", [0, 1])
@pytest.mark.parametrize("name", ["bidaf_small.pt", "bidaf_d200.pt"])
def test_backward_matches_reference_golden(name, precision):
    import torch.nn.functional as F
    g = load_golden(name)
    tol = BWD_TOL[precision]
    args = (g["state"], g["text"], g["modality"], g["text_mask"], g["modality_mask"], g["grad_out"])
    got = _grads(*args, precision=precision)
    _check_grads(got, g["grad_text"], g["grad_modality"], g["grad_params"], tol, _ds_abs_sum(*args) if precision else None)
    pr = g["train_drop_prob"]
    torch.manual_seed(g["train_seed"])
    keep_c = F.dropout(torch.ones_like(g["text"]), pr, True) != 0
    keep_q = F.dropout(torch.ones_like(g["modality"]), pr, True) != 0
    got = _grads(*args, keep_c, keep_q, pr, precision)
    _check_grads(got, g["train_grad_text"], g["train_grad_modality"], g["train_grad_params"], tol,
                 _ds_abs_sum(*args, keep_c, keep_q, pr) if precision else None)


@pytest.mark.parametrize("shape", [(1, 1, 1, 8), (2, 1, 9, 8), (2, 5, 3, 8), (3, 64, 128, 200), (2, 65, 129, 200),
                                   (2, 130, 257, 200), (4, 100, 70, 64), (2, 300, 520, 200), (3, 409, 1024, 200)])
@pytest.mark.parametrize("dropout", [False, True])
def test_bf16_backward_matches_oracle_ragged(shape, dropout):
    bsz, lc, lq, d = shape
    gen = torch.Generator().manual_seed(3000 + lc * 7 + lq)
    p = {"text_weight": torch.randn(d, 1, generator=gen) * 0.1, "modality_weight": torch.randn(d, 1, generator=gen) * 0.1,
         "text_modality_weight": torch.randn(1, 1, d, generator=gen) * 0.1, "bias": torch.tensor([0.3])}
    text = torch.randn(bsz, lc, d, generator=gen)
    modality = torch.randn(bsz, lq, d, generator=gen)
    c_len = torch.randint(1, lc + 1, (bsz,), generator=gen).tolist()
    q_len = torch.randint(1, lq + 1, (bsz,), generator=gen).tolist()
    c_len[0], q_len[0] = lc, lq
    tmask, mmask = O.length_mask(lc, c_len), O.length_mask(lq, q_len)
    grad_out = torch.randn(bsz, lc, 4 * d, generator=gen)
    pr = 0.2 if dropout else 0.0
    keep_c = (torch.rand(bsz, lc, d, generator=gen) >= pr) if dropout else None
    keep_q = (torch.rand(bsz, lq, d, generator=gen) >= pr) if dropout else None
    # fp64 oracle + autograd
    pd = {k: v.double().requires_grad_(True) for k, v in p.items()}
    cd, qd = text.double().requires_grad_(True), modality.double().requires_grad_(True)
    want = O.bidaf_attention(pd, cd, qd, tmask, mmask, keep_c, keep_q, pr)
    want.backward(grad_out.double())
    got = _grads(p, text, modality, tmask, mmask, grad_out, keep_c, keep_q, pr, precision=1)
    assert torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()
    # a soft-max over a single element has an identically zero gradient: with lc == 1 or lq == 1 some weight gradients
    # are pure cancellation noise (bf16: ~1e-3 of the terms that cancel), so their floor is set from the upstream scale
    w_floor = 5e-2 * float(grad_out.abs().sum()) if min(lc, lq) == 1 else 1e-3
    ds_scale = _ds_abs_sum(p, text, modality, tmask, mmask, grad_out, keep_c, keep_q, pr)
    _check_grads(got, cd.grad, qd.grad, {k: v.grad for k, v in pd.items()}, BWD_TOL[1], ds_scale, w_floor,
                 bias_slack=w_floor if min(lc, lq) == 1 else 0.0)


@pytest.mark.parametrize("shape", [(2, 130, 257, 200), (2, 600, 70, 200), (3, 409, 1024, 200)])
def test_bf16_tier_ragged_forward_backward(shape):
    """bf16 tier on ragged batches against the fp64 oracle: the forward with and without dropout, and the backward (through
    the saved state) with dropout."""
    bsz, lc, lq, d = shape
    gen = torch.Generator().manual_seed(4000 + lc * 7 + lq)
    p = {"text_weight": torch.randn(d, 1, generator=gen) * 0.1, "modality_weight": torch.randn(d, 1, generator=gen) * 0.1,
         "text_modality_weight": torch.randn(1, 1, d, generator=gen) * 0.1, "bias": torch.tensor([0.3])}
    text = torch.randn(bsz, lc, d, generator=gen)
    modality = torch.randn(bsz, lq, d, generator=gen)
    c_len = torch.randint(1, lc + 1, (bsz,), generator=gen).tolist()
    q_len = torch.randint(1, lq + 1, (bsz,), generator=gen).tolist()
    c_len[0], q_len[0] = lc, lq
    tmask, mmask = O.length_mask(lc, c_len), O.length_mask(lq, q_len)
    keep_c = torch.rand(bsz, lc, d, generator=gen) >= 0.2
    keep_q = torch.rand(bsz, lq, d, generator=gen) >= 0.2
    pd = {k: v.double() for k, v in p.items()}
    for kc, kq, pr in ((None, None, 0.0), (keep_c, keep_q, 0.2)):
        want = O.bidaf_attention(pd, text.double(), modality.double(), tmask, mmask, kc, kq, pr)
        out, *_ = _run(p, text, modality, tmask, mmask, kc, kq, pr, precision=1)
        assert torch.isfinite(out).all() and rel_err(out, want) < BF16_TOL
    grad_out = torch.randn(bsz, lc, 4 * d, generator=gen)
    pg = {k: v.double().requires_grad_(True) for k, v in p.items()}
    cd, qd = text.double().requires_grad_(True), modality.double().requires_grad_(True)
    O.bidaf_attention(pg, cd, qd, tmask, mmask, keep_c, keep_q, 0.2).backward(grad_out.double())
    got = _grads(p, text, modality, tmask, mmask, grad_out, keep_c, keep_q, 0.2, precision=1)
    _check_grads(got, cd.grad, qd.grad, {k: v.grad for k, v in pg.items()}, BWD_TOL[1],
                 _ds_abs_sum(p, text, modality, tmask, mmask, grad_out, keep_c, keep_q, 0.2))


@pytest.mark.parametrize("shape", [(1, 1, 1, 4), (2, 1, 9, 8), (2, 5, 3, 8), (3, 64, 32, 200), (2, 65, 33, 200), (2, 130, 257, 200),
                                   (4, 100, 70, 64), (2, 31, 95, 12)])
@pytest.mark.parametrize("dropout", [False, True])
def test_fp32_backward_matches_oracle_ragged(shape, dropout):
    """fp32 tier: the FFMA backward kernels (csrc/bidaf_bwd_f32.cu) against fp64 autograd of the oracle."""
    bsz, lc, lq, d = shape
    gen = torch.Generator().manual_seed(5000 + lc * 7 + lq)
    p = {"text_weight": torch.randn(d, 1, generator=gen) * 0.2, "modality_weight": torch.randn(d, 1, generator=gen) * 0.2,
         "text_modality_weight": torch.randn(1, 1, d, generator=gen) * 0.2, "bias": torch.tensor([0.3])}
    text = torch.randn(bsz, lc, d, generator=gen)
    modality = torch.randn(bsz, lq, d, generator=gen)
    c_len = torch.randint(1, lc + 1, (bsz,), generator=gen).tolist()
    q_len = torch.randint(1, lq + 1, (bsz,), generator=gen).tolist()
    c_len[0], q_len[0] = lc, lq
    tmask, mmask = O.length_mask(lc, c_len), O.length_mask(lq, q_len)
    grad_out = torch.randn(bsz, lc, 4 * d, generator=gen)
    pr = 0.2 if dropout else 0.0
    keep_c = (torch.rand(bsz, lc, d, generator=gen) >= pr) if dropout else None
    keep_q = (torch.rand(bsz, lq, d, generator=gen) >= pr) if dropout else None
    pd = {k: v.double().requires_grad_(True) for k, v in p.items()}
    cd, qd = text.double().requires_grad_(True), modality.double().requires_grad_(True)
    O.bidaf_attention(pd, cd, qd, tmask, mmask, keep_c, keep_q, pr).backward(grad_out.double())
    got = _grads(p, text, modality, tmask, mmask, grad_out, keep_c, keep_q, pr, precision=0)
    assert torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()
    # weight gradients that vanish analytically (soft-max over one element) are fp32 cancellation noise: floor them
    _check_grads(got, cd.grad, qd.grad, {k: v.grad for k, v in pd.items()}, BWD_TOL[0], None, 1e-2 if min(lc, lq) == 1 else 1e-3)


def test_backward_fully_masked_rows_match_oracle():
    """A fully masked soft-max is uniform (attention.py:94): its weights still carry dq, dT and R dT in the backward."""
    gen = torch.Generator().manual_seed(9)
    d, lc, lq = 8, 6, 5
    p = {"text_weight": torch.randn(d, 1, generator=gen), "modality_weight": torch.randn(d, 1, generator=gen),
         "text_modality_weight": torch.randn(1, 1, d, generator=gen), "bias": torch.tensor([0.0])}
    text, modality = torch.randn(2, lc, d, generator=gen), torch.randn(2, lq, d, generator=gen)
    tmask, mmask = O.length_mask(lc, [6, 0]), O.length_mask(lq, [0, 5])
    grad_out = torch.randn(2, lc, 4 * d, generator=gen)
    pd = {k: v.double().requires_grad_(True) for k, v in p.items()}
    cd, qd = text.double().requires_grad_(True), modality.double().requires_grad_(True)
    O.bidaf_attention(pd, cd, qd, tmask, mmask).backward(grad_out.double())
    for precision in (0, 1):
        dc, dq, dw = _grads(p, text, modality, tmask, mmask, grad_out, precision=precision)
        tol = BWD_TOL[precision]
        assert torch.isfinite(dc).all() and torch.isfinite(dq).all()
        assert grad_err(dc, cd.grad) < tol and grad_err(dq, qd.grad) < tol, (precision, grad_err(dc, cd.grad), grad_err(dq, qd.grad))


def test_full_size_config2_tiers_agree_and_backward_is_linear():
    """BASELINE config 2 at full size (B=64, Lc=512, Lq=256, d=200), where the CPU oracle is too slow: the tensor-core tier
    against the fp32 tier (itself pinned to the oracle at small sizes), forward and backward, plus two size-independent
    properties: the backward is linear in the upstream gradient, and padded modality rows get exactly zero gradient."""
    from mmbidaf_b200 import functional as F
    bsz, lc, lq, d = 64, 512, 256, 200
    gen = torch.Generator().manual_seed(224)
    c = torch.randn(bsz, lc, d, generator=gen).cuda()
    q = torch.randn(bsz, lq, d, generator=gen).cuda()
    c_len = torch.randint(lc // 2, lc + 1, (bsz,), generator=gen)
    q_len = torch.randint(lq // 2, lq + 1, (bsz,), generator=gen)
    c_len[0], q_len[0] = lc, lq
    tmask = (torch.arange(lc).unsqueeze(0) < c_len.unsqueeze(1)).cuda()
    mmask = (torch.arange(lq).unsqueeze(0) < q_len.unsqueeze(1)).cuda()
    w = [(torch.randn(d, generator=gen) * 0.1).cuda() for _ in range(3)]
    bias = torch.full((1,), 0.3).cuda()
    g1 = torch.randn(bsz, lc, 4 * d, generator=gen).cuda()
    g2 = torch.randn(bsz, lc, 4 * d, generator=gen).cuda()

    def run(precision, grad):
        leaves = [c.clone().requires_grad_(True), q.clone().requires_grad_(True)] + [t.clone().requires_grad_(True) for t in w]
        out = F.bidaf_attention(leaves[0], leaves[1], tmask, mmask, leaves[2].view(d, 1), leaves[3].view(d, 1),
                                leaves[4].view(1, 1, d), bias, None, None, 1.0, precision)
        out.backward(grad)
        return out.detach(), [t.grad for t in leaves]

    out32, grads32 = run(0, g1)
    out16, grads16 = run(1, g1)
    assert rel_err(out16, out32) < BF16_TOL
    for a, b in zip(grads16, grads32):
        assert grad_err(a, b) < BWD_TOL[1]
    # linearity of the backward pass in the upstream gradient (exact in exact arithmetic)
    _, ga = run(1, g1)
    _, gb = run(1, g2)
    _, gab = run(1, 0.5 * g1 + g2)
    for x, y, z in zip(ga, gb, gab):
        assert grad_err(z, 0.5 * x + y) < 2e-2
    # padded modality rows are masked out of s1 and never reach the output: their gradient is exactly zero
    dq = grads16[1]
    for b_, n in enumerate(q_len.tolist()):
        if n < lq:
            assert (dq[b_, n:] == 0).all()


def test_bf16_inference_path_writes_only_out():
    """aux=False (what the layer runs under no_grad): T and the log-sum-exps are neither allocated nor written; `out` is bit-identical
    to the full call."""
    from mmbidaf_b200 import ops
    gen = torch.Generator().manual_seed(99)
    c, q = torch.randn(3, 140, 200, generator=gen).cuda(), torch.randn(3, 75, 200, generator=gen).cuda()
    cm = (torch.arange(140).unsqueeze(0) < torch.tensor([[140], [17], [90]])).cuda()
    qm = (torch.arange(75).unsqueeze(0) < torch.tensor([[75], [75], [3]])).cuda()
    w = [(torch.randn(200, generator=gen) * 0.1).cuda() for _ in range(3)]
    bias = torch.tensor([0.2]).cuda()
    full = ops.bidaf_fwd(c, q, cm, qm, w[0], w[1], w[2], bias, precision=ops.PREC_BF16)
    lean = ops.bidaf_fwd(c, q, cm, qm, w[0], w[1], w[2], bias, precision=ops.PREC_BF16, aux=False)
    assert lean[1] is None and lean[2] is None and lean[3] is None
    assert torch.equal(full[0], lean[0])
