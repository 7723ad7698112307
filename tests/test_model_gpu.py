"""GPU parity of the whole path: mmbidaf_b200.models.MMBiDAF vs the reference's golden outputs."""
import pytest
import torch

from conftest import grad_err, load_golden, rel_err
from mmbidaf_b200.synth import Batch, make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _model(dims, params, drop=0.0):
    from mmbidaf_b200.models import MMBiDAF
    hidden, e_t, e_a, e_i, m = dims
    model = MMBiDAF(hidden, e_t, e_a, e_i, torch.device("cuda"), drop_prob=drop, max_transcript_length=m)
    missing, unexpected = model.load_state_dict(params, strict=True)
    assert not missing and not unexpected
    return model.cuda()


def _call(model, batch, train):
    model.train(train)
    model.zero_grad()
    b = batch.to("cuda")
    out, loss = model(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, b.targets, b.target_len,
                      b.max_dec_len)
    return out, loss


def test_small_model_matches_reference_golden():
    g = load_golden("model_small.pt")
    model = _model(g["dims"], g["params"])
    batch = Batch(**g["batch"])
    out, loss = _call(model, batch, True)
    assert rel_err(out, g["train_out"]) < TOL and rel_err(loss, g["train_loss"]) < TOL
    loss.backward()
    for name, p in model.named_parameters():
        if name in g["train_grads"]:
            assert grad_err(p.grad, g["train_grads"][name], name) < 2e-4, name
    with torch.no_grad():
        out_e, loss_e = _call(model, batch, False)
    assert rel_err(out_e, g["eval_out"]) < TOL and rel_err(loss_e, g["eval_loss"]) < TOL
    assert torch.equal(out_e.argmax(dim=2).cpu(), g["eval_argmax"])            # selected sentence indices


def test_readme_size_model_matches_reference_golden():
    g = load_golden("model_readme.pt")
    hidden, e_t, e_a, e_i, m = g["dims"]
    params = O.make_params(hidden, e_t, e_a, e_i, m, seed=g["param_seed"])
    model = _model(g["dims"], params)
    batch = make_batch(*g["batch_shape"], e_t, e_a, e_i, seed=g["batch_seed"])
    out, loss = _call(model, batch, True)
    assert rel_err(out, g["train_out"]) < TOL and rel_err(loss, g["train_loss"]) < TOL
    loss.backward()
    grads = dict(model.named_parameters())
    for name, want in g["train_grads_sample"].items():
        assert grad_err(grads[name].grad, want, name) < 2e-4, name
    for name, want in g["train_grad_norms"].items():
        got = float(grads[name].grad.double().norm())
        assert abs(got - want) <= 2e-3 * max(want, 1e-3), name   # tiny norms are cancellation noise
    with torch.no_grad():
        out_e, loss_e = _call(model, batch, False)
    assert rel_err(out_e, g["eval_out"]) < TOL and rel_err(loss_e, g["eval_loss"]) < TOL
    assert torch.equal(out_e.argmax(dim=2).cpu(), g["eval_argmax"])
    # greedy extractive decoding (evaluate.py:185-202): identical index lists
    from mmbidaf_b200.decode import get_generated_indices
    want = [O.greedy_indices(g["eval_out"][b], batch.text_len[b]) for b in range(len(batch.text_len))]
    assert get_generated_indices(out_e, batch.text_len) == want


def test_accepts_dataparallel_checkpoint_and_masks_bit_exact():
    g = load_golden("model_small.pt")
    model = _model(g["dims"], {"module." + k: v for k, v in g["params"].items()})
    batch = Batch(**g["batch"])
    x = batch.text.cuda()
    assert torch.equal(model.get_mask(x, batch.text_len).cpu(), O.length_mask(x.shape[1], batch.text_len))


def test_masked_softmax_function_matches_reference_golden():
    from mmbidaf_b200.layers import masked_softmax
    g = load_golden("masked_softmax.pt")
    cu = lambda t: t.cuda()
    assert rel_err(masked_softmax(cu(g["logits"]), cu(g["row_mask"]), dim=2), g["row"]) < TOL
    assert rel_err(masked_softmax(cu(g["logits"]), cu(g["col_mask"]), dim=1), g["col"]) < TOL
    assert rel_err(masked_softmax(cu(g["flat"]), cu(g["flat_mask"])), g["flat_out"]) < TOL
    got_log = masked_softmax(cu(g["flat"]), cu(g["flat_mask"]), log_softmax=True)
    assert rel_err(got_log, g["flat_log"]) < TOL
    x = g["flat"].cuda().requires_grad_(True)
    xr = g["flat"].clone().requires_grad_(True)
    w = torch.randn(3, 9)
    (masked_softmax(x, cu(g["flat_mask"])) * w.cuda()).sum().backward()
    (O.masked_softmax(xr, g["flat_mask"]) * w).sum().backward()
    assert grad_err(x.grad, xr.grad) < TOL


def test_streams_do_not_change_results():
    g = load_golden("model_small.pt")
    batch = Batch(**g["batch"])
    outs = []
    for use in (True, False):
        model = _model(g["dims"], g["params"])
        model.use_streams = use
        out, loss = _call(model, batch, True)
        loss.backward()
        torch.cuda.synchronize()
        outs.append((out.detach().clone(), loss.detach().clone(), model.emb.proj.weight.grad.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_dropout_keys_do_not_depend_on_stream_timing():
    """Training with dropout: the encoder chains run on side streams, but which layer gets which dropout key must not depend on
    when the GPU gets to each chain.  Holding the text chain's stream back (so that the image chain draws its keys first when the
    draws follow the GPU's order) leaves the output and the loss bit for bit the same."""
    from mmbidaf_b200 import ops
    from mmbidaf_b200.models import MMBiDAF
    torch.manual_seed(3)
    model = MMBiDAF(100, 300, 128, 1000, torch.device("cuda"), drop_prob=0.2, max_transcript_length=64).cuda()
    batch = make_batch(4, 40, 90, 11, 5, seed=31)

    def run(delay_text):
        ops.rng_seed(11)
        if delay_text:
            with torch.cuda.stream(model._streams[1]):                 # (audio, text, image)
                torch.cuda._sleep(50_000_000)                          # ~25 ms
        out, loss = _call(model, batch, True)
        torch.cuda.synchronize()
        return out.detach().clone(), loss.detach().clone()

    want = run(False)
    got = run(True)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_tf32_library_gemms_stay_inside_the_reduced_precision_tier():
    """north_star: rel <= 2e-2 on the TF32/bf16 path.  Only the plain library GEMMs change here."""
    g = load_golden("model_readme.pt")
    hidden, e_t, e_a, e_i, m = g["dims"]
    params = O.make_params(hidden, e_t, e_a, e_i, m, seed=g["param_seed"])
    model = _model(g["dims"], params)
    batch = make_batch(*g["batch_shape"], e_t, e_a, e_i, seed=g["batch_seed"])
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        out, loss = _call(model, batch, True)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    assert rel_err(out, g["train_out"]) < 2e-2 and rel_err(loss, g["train_loss"]) < 2e-2


def test_fast_tier_whole_model_within_reduced_precision_tolerance():
    """set_precision('fast'): tcgen05 bf16 BiDAF + TF32 library GEMMs; north_star rel <= 2e-2."""
    import mmbidaf_b200
    g = load_golden("model_readme.pt")
    hidden, e_t, e_a, e_i, m = g["dims"]
    params = O.make_params(hidden, e_t, e_a, e_i, m, seed=g["param_seed"])
    model = _model(g["dims"], params)
    batch = make_batch(*g["batch_shape"], e_t, e_a, e_i, seed=g["batch_seed"])
    mmbidaf_b200.set_precision("fast")
    try:
        out, loss = _call(model, batch, True)
        loss.backward()
        torch.cuda.synchronize()
        grads = dict(model.named_parameters())
        assert rel_err(out, g["train_out"]) < 2e-2 and rel_err(loss, g["train_loss"]) < 2e-2
        for name, want in g["train_grads_sample"].items():
            assert grad_err(grads[name].grad, want, name) < 5e-2, name
        with torch.no_grad():
            out_e, _ = _call(model, batch, False)
        assert rel_err(out_e, g["eval_out"]) < 2e-2
    finally:
        mmbidaf_b200.set_precision("fp32")


def test_embedding_highway_matches_reference_golden():
    from mmbidaf_b200.layers import Embedding
    g = load_golden("embedding.pt")
    mod = Embedding(embedding_size=10, hidden_size=6, drop_prob=0.0)
    mod.load_state_dict(g["state"])
    mod = mod.cuda().eval()
    x = g["x"].cuda().requires_grad_(True)
    out = mod(x)
    assert rel_err(out, g["out"]) < TOL
    # gradients against the oracle's autograd
    w = torch.randn(2, 5, 6)
    (out * w.cuda()).sum().backward()
    p = {k: v.clone().requires_grad_(True) for k, v in g["state"].items()}
    xr = g["x"].clone().requires_grad_(True)
    (O.embedding(p, xr) * w).sum().backward()
    assert grad_err(x.grad, xr.grad) < 1e-5
    for name, param in mod.named_parameters():
        assert grad_err(param.grad, p[name].grad, name) < 1e-5, name
