"""GPU: every way the launchers of the decoder kernels can run a step, against the fp64 oracle (oracle.mmbidaf_oracle.decoder_step).

The cluster kernels (csrc/decoder_fused.cu) read a CTA's text rows of proj_* / enc_* either from a ROW STAGE in shared memory (bulk
copies) or straight from L2.  launch_fused (forward step and every roll-out) and mmb_decoder_step_fused_bwd take the stage only when
D % 4 == 0, the row pointers are 16-byte aligned, the stage fits in 227 KB of shared memory and MMB_DEC_STAGE is not 0.  The weighted
contexts of the forward (both cuts) read enc_* as float4 only when D % 4 == 0 and enc_* are 16-byte aligned, one float at a time
otherwise.  Cluster size: 8 CTAs when B * 8 <= 160, else 4; chunk = ceil(Lt / cluster) text rows per CTA; D = 2 * hidden.

Each case below forces its path by construction, not by today's shared-memory margins -- except config 3, which is here because the
benchmark runs it:

  case            (B, Lt, hidden, E, M)    path            why
  staged-8cta     (3, 24, 100, 300, 409)   staged          8 CTAs, chunk 3: stage chunk * D * 8 = 4 800 B <= 64 KB
  config3-4cta    (32, 409, 100, 300, 409) staged          4 CTAs, chunk 103: stage 164 800 B; forward 216.5 KB, backward 222.0 KB
                                                           of 227 KB in all (a margin: a layout change can move it to L2)
  l2size-4cta     (32, 600, 100, 300, 600) L2 by size      4 CTAs, chunk 150: stage 240 000 B > 232 448 B on its own;
                                                           B * Lt = 19 200 <= 20 000: the fused cut by default (training at Lt 600)
  l2size-8cta     (16, 1250, 100, 300, 1250) L2 by size    8 CTAs, chunk 157: 251 200 B > 232 448 B; B * Lt = 20 000: fused
  long-lecture    (2, 4096, 100, 300, 4096) L2 by size     8 CTAs, chunk 512: 819 200 B
  empty-ranks     (21, 3, 100, 300, 9)     staged          4 CTAs (21 * 8 = 168 > 160), chunk 1: rank 3 has no text rows
  odd-8cta        (5, 37, 33, 10, 40)      L2 by width     D = 66 = 2 (mod 4): no stage, scalar context loop, scalar mat-vecs
  odd-4cta        (21, 500, 33, 300, 500)  L2 by width     D = 66 on a 4-CTA cluster, chunk 125
  d194            (3, 50, 97, 300, 64)     L2 by width     D = 194: seven column registers (192 < D <= 224), scalar context loop
  d256            (4, 40, 128, 300, 64)    staged          D = 256, the largest allowed: all eight column registers used

and two paths that take inputs rather than shapes:

  L2 by alignment  enc_a / enc_i copied into buffers at a one-float offset (4-byte aligned rows): test_unaligned_*
  L2 by switch     MMB_DEC_STAGE=0, read once per process on the first launch, so set in a child process: test_stage_off_*
"""
import os
import subprocess
import sys

import pytest
import torch

from conftest import grad_err, rel_err
from oracle import mmbidaf_oracle as O
from test_beam_gpu import _reference as _beam_reference

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
TOL = 1e-5
STEPS = 3            # chained steps of the backward tests

CASES = {
    "staged-8cta": ((3, 24, 100, 300, 409), "staged"),
    "config3-4cta": ((32, 409, 100, 300, 409), "staged"),
    "l2size-4cta": ((32, 600, 100, 300, 600), "L2 by size"),
    "l2size-8cta": ((16, 1250, 100, 300, 1250), "L2 by size"),
    "long-lecture": ((2, 4096, 100, 300, 4096), "L2 by size"),
    "empty-ranks": ((21, 3, 100, 300, 9), "staged"),
    "odd-8cta": ((5, 37, 33, 10, 40), "L2 by width"),
    "odd-4cta": ((21, 500, 33, 300, 500), "L2 by width"),
    "d194": ((3, 50, 97, 300, 64), "L2 by width"),
    "d256": ((4, 40, 128, 300, 64), "staged"),
}
L2_BY_SIZE = [c for c, (_, path) in CASES.items() if path == "L2 by size"]
ODD = ["odd-8cta", "odd-4cta"]


def _make(case):
    """A decoder module with seeded weights (uniform in +-0.2, as test_decoder_step_matches_oracle) and seeded inputs on the device:
    (module, inputs, text lengths (B) int64, mask (B, M) bool, targets (8, B) int64 inside each video's length)."""
    from mmbidaf_b200.layers import MultimodalAttentionDecoder
    bsz, lt, hid, e, m = CASES[case][0]
    gen = torch.Generator().manual_seed(4000 + 7 * bsz + lt + hid)
    mod = MultimodalAttentionDecoder(e, hid, m, num_layers=1)
    mod.load_state_dict({k: (torch.rand(v.shape, generator=gen) - 0.5) * 0.4 for k, v in mod.state_dict().items()})
    mod = mod.cuda()
    d = 2 * hid
    x = {"enc_a": torch.randn(bsz, lt, d, generator=gen), "enc_i": torch.randn(bsz, lt, d, generator=gen),
         "h": torch.randn(bsz, hid, generator=gen), "cell": torch.randn(bsz, hid, generator=gen), "cov": torch.rand(bsz, lt, generator=gen),
         "sents": torch.randn(STEPS, bsz, e, generator=gen), "emb": torch.randn(bsz, lt, e, generator=gen)}
    x = {k: v.cuda() for k, v in x.items()}
    lens = torch.randint(1, lt + 1, (bsz,), generator=gen)
    lens[0] = lt                                                          # one video uses every text row
    mask = (torch.arange(m).unsqueeze(0) < lens.unsqueeze(1)).cuda()
    tgts = torch.stack([torch.stack([torch.randint(0, int(n), (1,), generator=gen)[0] for n in lens]) for _ in range(8)]).cuda()
    return mod, x, lens.cuda(), mask, tgts


def _seq(mod, enc_a, enc_i):
    with torch.no_grad():
        return mod._sequence(enc_a, enc_i)["seq"]


def _p64(mod):
    return {k: v.detach().double() for k, v in mod.state_dict().items()}


def _oracle_step(mod, x, mask, enc_a=None, enc_i=None):
    """O.decoder_step in float64 on the device: (probs, h', cell', att_cov, coverage') as (B, M), (B, H), (B, H), (B, Lt), (B, Lt)."""
    d64 = lambda t: t.detach().double()
    enc_a = x["enc_a"] if enc_a is None else enc_a
    enc_i = x["enc_i"] if enc_i is None else enc_i
    out = O.decoder_step(_p64(mod), d64(x["sents"][0]).unsqueeze(1), d64(x["h"]).unsqueeze(1), d64(x["cell"]).unsqueeze(0), d64(enc_a),
                         d64(enc_i), d64(x["cov"]).unsqueeze(2), mask)
    return out[0], out[1].squeeze(1), out[2].squeeze(0), out[3].squeeze(2), out[4].squeeze(2)


def _step(seq, x, mask, target=None):
    from mmbidaf_b200 import ops
    out = ops.decoder_step_fwd(seq, x["sents"][0], x["h"], x["cell"], x["cov"], mask.to(torch.uint8), want_argmax=True, target=target)
    torch.cuda.synchronize()
    return out


def _clear_rows(probs):
    """Rows whose oracle arg-max is decided: top-two gap at least 1e-6 of the top value."""
    top = probs.topk(2, dim=1).values
    return (top[:, 0] - top[:, 1]) >= 1e-6 * top[:, 0]


def _check_step_against_oracle(got, want, mask, what):
    errs = {name: rel_err(g, w) for name, g, w in zip(("probs", "h", "cell", "att_cov", "coverage"), got[:5], want)}
    assert max(errs.values()) < TOL, (what, errs)
    clear = _clear_rows(want[0])
    assert clear.any(), what
    assert torch.equal(got[5][clear], want[0].argmax(dim=1)[clear]), what               # the selected sentence: exact
    assert (got[0][~mask] == 0).all(), what                                             # no mass past a video's length
    assert (got[0].sum(dim=1) - 1).abs().max() < 1e-5, what


@pytest.mark.parametrize("case", list(CASES))
def test_forward_step_matches_the_fp64_oracle(case, monkeypatch):
    """One step on both cuts -- the cluster kernel (staged or L2 as the case forces) and the chunk-parallel cut -- against the oracle:
    every output within 1e-5, the arg-max exact where the oracle's top two are apart, zero probability past each video's length."""
    mod, x, _, mask, _ = _make(case)
    want = _oracle_step(mod, x, mask)
    seq = _seq(mod, x["enc_a"], x["enc_i"])
    for cut in ("fused", "chunks"):
        monkeypatch.setenv("MMB_DECODER_CUT", cut)
        _check_step_against_oracle(_step(seq, x, mask), want, mask, cut)


def _chain(mod, x, mask, tgts, fused_loss, enc_a, enc_i, steps=STEPS):
    """``steps`` chained training steps through the module from h0 = x["h"] (a leaf here), then backward.  fused_loss: the kernels'
    loss terms (target=); else the same terms composed with torch ops plus sum p^2, so that d probs is dense.
    Returns (loss, d h0, {name: parameter gradient})."""
    mod.train()
    mod.zero_grad(set_to_none=True)
    h = x["h"].clone().requires_grad_(True)
    state = (h.unsqueeze(1), x["cell"].unsqueeze(0), x["cov"].unsqueeze(2))
    loss = 0
    for k in range(steps):
        sent = x["sents"][k].unsqueeze(1)
        if fused_loss:
            probs, h1, c1, att, cov, terms = mod.step(sent, state[0], state[1], enc_a, enc_i, state[2], mask, target=tgts[k])
            loss = loss + terms.sum()
        else:
            probs, h1, c1, att, cov = mod(sent, state[0], state[1], enc_a, enc_i, state[2], mask)
            loss = (loss - torch.log(probs.gather(1, tgts[k].unsqueeze(1)) + 1e-12).sum() + torch.min(att, cov).sum()
                    + (probs * probs).sum())
        state = (h1, c1, cov)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), h.grad, {n: p.grad for n, p in mod.named_parameters()}


def _oracle_chain(mod, x, mask, tgts, fused_loss):
    """The same chain through O.decoder_step in float64 with the module's state_dict as leaves: (loss, d enc_a, d enc_i, d h0, grads)."""
    p = {k: v.requires_grad_(True) for k, v in _p64(mod).items()}
    enc_a = x["enc_a"].double().requires_grad_(True)
    enc_i = x["enc_i"].double().requires_grad_(True)
    h0 = x["h"].double().requires_grad_(True)
    h, cell, cov = h0.unsqueeze(1), x["cell"].double().unsqueeze(0), x["cov"].double().unsqueeze(2)
    loss = 0
    for k in range(STEPS):
        probs, h, cell, att, cov = O.decoder_step(p, x["sents"][k].double().unsqueeze(1), h, cell, enc_a, enc_i, cov, mask)
        loss = loss - torch.log(probs.gather(1, tgts[k].unsqueeze(1)) + 1e-12).sum() + torch.min(att, cov).sum()
        if not fused_loss:
            loss = loss + (probs * probs).sum()
    loss.backward()
    return loss.detach(), enc_a.grad, enc_i.grad, h0.grad, {k: v.grad for k, v in p.items()}


def _grad_errs(got_loss, got_a, got_i, got_h, got_p, want):
    want_loss, want_a, want_i, want_h, want_p = want
    errs = {"loss": rel_err(got_loss, want_loss), "enc_a": grad_err(got_a, want_a), "enc_i": grad_err(got_i, want_i),
            "h0": grad_err(got_h, want_h)}
    errs.update({n: grad_err(g, want_p[n], n) for n, g in got_p.items()})
    return errs


def _grad_tol(name):
    # v_beta_1 / v_beta_2 bias gradients: beta_k (db_k - mix), a difference of nearly equal sums over the text axis -- cancellation noise
    # at the 1e-4 level (as in test_decoder_gpu.py); v1 / v2 bias gradients are identically zero (grad_err checks them as such)
    return 5e-4 if name in ("v_beta_1.bias", "v_beta_2.bias") else 5e-5


@pytest.mark.parametrize("fused_loss", [True, False])
@pytest.mark.parametrize("case", list(CASES))
def test_backward_matches_fp64_autograd(case, fused_loss, monkeypatch):
    """Three chained steps through MultimodalAttentionDecoder and autograd (the whole backward step as one cluster kernel, staged or L2
    as the case forces; on the L2-by-size shapes also the chunk-parallel cut) against fp64 autograd through the oracle: d enc_a, d enc_i,
    d h0 and every parameter gradient."""
    mod, x, _, mask, tgts = _make(case)
    want = _oracle_chain(mod, x, mask, tgts, fused_loss)
    for cut in ("fused", "chunks") if case in L2_BY_SIZE else ("fused",):
        monkeypatch.setenv("MMB_DECODER_CUT", cut)
        enc_a = x["enc_a"].clone().requires_grad_(True)
        enc_i = x["enc_i"].clone().requires_grad_(True)
        loss, d_h, grads = _chain(mod, x, mask, tgts, fused_loss, enc_a, enc_i)
        errs = _grad_errs(loss, enc_a.grad, enc_i.grad, d_h, grads, want)
        bad = {n: e for n, e in errs.items() if e >= (TOL if n == "loss" else _grad_tol(n))}
        assert not bad, (cut, bad)


# ---- MMB_DEC_STAGE=0 in a child process: the L2 arm on exactly the inputs the parent runs staged --------------------------------------

STAGE_CASES = ["staged-8cta", "config3-4cta"]


def _stage_outputs(case):
    """Everything the row stage feeds, on the case's seeded inputs: one forward step (outputs and saved state), two training steps
    through the module (one with the fused loss terms, one with a dense d probs) and their gradients, a greedy roll-out with loss terms
    and a beam roll-out of width 3.  Runs the cluster kernels (MMB_DECODER_CUT=fused in both processes)."""
    mod, x, lens, mask, tgts = _make(case)
    out = {}
    fwd = _step(_seq(mod, x["enc_a"], x["enc_i"]), x, mask, target=tgts[0])
    for name, t in zip(("probs", "h", "cell", "att_cov", "coverage", "argmax"), fwd[:6]):
        out[f"step.{name}"] = t
    for name, t in zip(("hw", "alpha", "beta", "ctx12", "pb", "xcat", "gates"), fwd[6]):
        out[f"step.saved.{name}"] = t
    out["step.loss_terms"] = fwd[7]
    enc_a = x["enc_a"].clone().requires_grad_(True)
    enc_i = x["enc_i"].clone().requires_grad_(True)
    mod.train()
    mod.zero_grad(set_to_none=True)
    h = x["h"].clone().requires_grad_(True)
    s0 = x["sents"][0].unsqueeze(1)
    probs, h1, c1, att, cov, terms = mod.step(s0, h.unsqueeze(1), x["cell"].unsqueeze(0), enc_a, enc_i, x["cov"].unsqueeze(2), mask,
                                              target=tgts[0])
    probs, _, _, att, cov = mod(x["sents"][1].unsqueeze(1), h1, c1, enc_a, enc_i, cov, mask)
    loss = terms.sum() + (probs * probs).sum() + torch.min(att, cov).sum()
    loss.backward()
    out.update({"bwd.loss": loss.detach(), "bwd.enc_a": enc_a.grad, "bwd.enc_i": enc_i.grad, "bwd.h0": h.grad})
    out.update({f"bwd.{n}": p.grad for n, p in mod.named_parameters()})
    mod.eval()
    g_probs, g_picks, g_terms = mod.greedy(x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, 8, target=tgts.t().contiguous())
    out.update({"greedy.probs": g_probs, "greedy.picks": g_picks, "greedy.loss_terms": g_terms})
    for name, t in zip(("tokens", "parents", "scores", "probs", "best", "path"),
                       mod.beam(x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, lens, 6, 3)):
        out[f"beam.{name}"] = t
    torch.cuda.synchronize()
    return {k: v.detach().cpu() for k, v in out.items()}


def _stage_child(path, case):
    """Entry point of the child process (MMB_DEC_STAGE=0 in its environment)."""
    torch.save(_stage_outputs(case), path)


@pytest.mark.parametrize("case", STAGE_CASES)
def test_stage_off_is_bit_identical(case, tmp_path, monkeypatch):
    """The same seeded work with the row stage (this process) and without it (a child with MMB_DEC_STAGE=0): bit for bit.  Why it
    holds: the energies' rows are independent of the warps' row grouping (2 rows per warp iteration staged, 4 from L2); the context
    partials take the same float4 loop on both arms; the backward's column partials add the warps in the same order (staged: two
    passes of 8 warps, L2: one pass of 16); d proj has one writer per element and step (a bulk reduction staged, a red.add from L2);
    and the backward's mat-vec scratch (halved when staged) still holds NT / (n_out / 4) K slices for every n_out when D >= 86, so the
    slice count -- the summation order -- is the same (D = 200 here)."""
    if os.environ.get("MMB_DEC_STAGE", "").strip() == "0":
        pytest.skip("MMB_DEC_STAGE=0 in this process: nothing runs staged to compare with")
    off_path = tmp_path / "stage_off.pt"
    env = dict(os.environ, MMB_DEC_STAGE="0", MMB_DECODER_CUT="fused")
    code = ("import sys; sys.path[:0] = sys.argv[1:3]; import test_decoder_paths_gpu as t; t._stage_child(sys.argv[3], sys.argv[4])")
    args = [sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", code, TESTS, ROOT, str(off_path), case]
    res = subprocess.run(args, env=env, cwd=ROOT, timeout=900, capture_output=True, text=True)
    assert res.returncode == 0, (res.stdout[-2000:], res.stderr[-4000:])
    off = torch.load(off_path, weights_only=True)
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    on = _stage_outputs(case)
    assert set(on) == set(off)
    differ = [k for k in on if not torch.equal(on[k], off[k])]
    assert not differ, differ


# ---- enc_a / enc_i at a 4-byte offset: the L2 arm with the scalar context loop ------------------------------------------------------

UNALIGNED_CASES = ["staged-8cta", "l2size-4cta"]


def _unaligned(t):
    """A copy of ``t`` that starts one float into its buffer: rows 4-byte but not 16-byte aligned.  Returns (view, buffer)."""
    buf = torch.zeros(t.numel() + 1, device=t.device, dtype=t.dtype)
    buf[1:].copy_(t.reshape(-1))
    view = buf[1:].view(t.shape)
    assert view.data_ptr() % 16 == 4
    return view, buf


@pytest.mark.parametrize("case", UNALIGNED_CASES)
def test_unaligned_encoder_rows_forward(case, monkeypatch):
    """A step, the greedy roll-out and the beam roll-out (width 3) on unaligned enc_a / enc_i, on both cuts: within 1e-6 of the aligned
    run (not bit for bit: the scalar context loop splits the rows over the threads differently) and the step within 1e-5 of the oracle."""
    mod, x, lens, mask, _ = _make(case)
    ua, _ = _unaligned(x["enc_a"])
    ui, _ = _unaligned(x["enc_i"])
    want = _oracle_step(mod, x, mask)
    mod.eval()
    for cut in ("fused", "chunks"):
        monkeypatch.setenv("MMB_DECODER_CUT", cut)
        ref = _step(_seq(mod, x["enc_a"], x["enc_i"]), x, mask)
        got = _step(_seq(mod, ua, ui), x, mask)
        _check_step_against_oracle(got, want, mask, cut)
        errs = {name: rel_err(g, r) for name, g, r in zip(("probs", "h", "cell", "att_cov", "coverage"), got[:5], ref[:5])}
        errs.update({f"saved.{name}": rel_err(g, r) for name, g, r in zip(("hw", "alpha", "beta", "ctx12", "pb", "xcat", "gates"),
                                                                           got[6], ref[6])})
        assert max(errs.values()) < 1e-6, (cut, errs)
        assert torch.equal(got[5], ref[5]), cut
        g_ref = mod.greedy(x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, 8)
        g_got = mod.greedy(x["emb"], x["h"], ua, ui, mask, 8)
        assert torch.equal(g_got[1], g_ref[1]), cut
        assert rel_err(g_got[0], g_ref[0]) < 1e-6, cut
    b_ref = mod.beam(x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, lens, 6, 3)
    b_got = mod.beam(x["emb"], x["h"], ua, ui, mask, lens, 6, 3)
    for name, g, r in zip(("tokens", "parents", "best", "path"), (b_got[0], b_got[1], b_got[4], b_got[5]),
                          (b_ref[0], b_ref[1], b_ref[4], b_ref[5])):
        assert torch.equal(g, r), name
    live = torch.isfinite(b_ref[2])
    assert torch.equal(live, torch.isfinite(b_got[2]))
    assert rel_err(b_got[2][live], b_ref[2][live]) < 1e-6 and rel_err(b_got[3], b_ref[3]) < 1e-6


@pytest.mark.parametrize("fused_loss", [True, False])
@pytest.mark.parametrize("case", UNALIGNED_CASES)
def test_unaligned_encoder_rows_backward_step_is_bit_identical(case, fused_loss, monkeypatch):
    """One backward step (ops.decoder_step_bwd) from the same saved forward state and incoming gradients, once over aligned and once
    over unaligned enc_a / enc_i (same proj rows): bit for bit on both cuts.  The backward reads enc rows one float per lane on every
    arm, so only the arm changes (staged-8cta: staged -> L2), and the arms agree bit for bit (test_stage_off_is_bit_identical)."""
    from mmbidaf_b200 import ops
    from mmbidaf_b200.layers.attention import _lib_fields
    mod, x, _, mask, tgts = _make(case)
    B, Lt, D = x["enc_a"].shape
    H, M = mod.hidden_size, mod.output_size
    with torch.no_grad():
        w = ops.DecoderWeights({f: mod._param_of(f) for f in _lib_fields()}, M)
        proj_a = torch.addmm(mod.W1.bias, x["enc_a"].view(-1, D), mod.W1.weight.t()).view(B, Lt, D)
        proj_i = torch.addmm(mod.W3.bias, x["enc_i"].view(-1, D), mod.W3.weight.t()).view(B, Lt, D)
    ua, _ = _unaligned(x["enc_a"])
    ui, _ = _unaligned(x["enc_i"])
    seqs = [ops.DecoderSeq(None, ea, ei, proj_a, proj_i, M, weights=w) for ea, ei in ((x["enc_a"], x["enc_i"]), (ua, ui))]
    assert seqs[1].enc_a.data_ptr() % 16 == 4
    gen = torch.Generator(device="cuda").manual_seed(31)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    grads_in = {"d_probs": None if fused_loss else rnd(B, M), "d_h_out": rnd(B, H), "d_cell_out": rnd(B, H), "d_att_cov": rnd(B, Lt),
                "d_cov_out": rnd(B, Lt), "d_lossvec": rnd(2, B) if fused_loss else None}
    mask_u8 = mask.to(torch.uint8)
    for cut in ("fused", "chunks"):
        monkeypatch.setenv("MMB_DECODER_CUT", cut)
        fwd = ops.decoder_step_fwd(seqs[0], x["sents"][0], x["h"], x["cell"], x["cov"], mask_u8, target=tgts[0])
        outs = []
        for seq in seqs:
            acc = [torch.zeros(B, Lt, D, device="cuda"), torch.zeros(B, Lt, D, device="cuda"), torch.zeros(B, 6, D, device="cuda"),
                   torch.zeros(B, 4, device="cuda")]
            res = ops.decoder_step_bwd(seq, x["h"], x["cell"], x["cov"], fwd[0], fwd[2], fwd[6], grads_in["d_probs"], grads_in["d_h_out"],
                                       grads_in["d_cell_out"], grads_in["d_att_cov"], grads_in["d_cov_out"], *acc,
                                       target=tgts[0] if fused_loss else None, d_lossvec=grads_in["d_lossvec"], att_cov=fwd[3],
                                       cov_out=fwd[4])
            torch.cuda.synchronize()
            outs.append([*res, *acc])
        names = ("d_h", "d_cell", "d_cov", "d_logits", "d_gates", "d_ctx12", "d_hw4", "d_pre_b", "d_proj_a", "d_proj_i", "vec_acc",
                 "scal_acc")
        differ = [n for n, a, u in zip(names, *outs) if not torch.equal(a, u)]
        assert not differ, (cut, differ)


@pytest.mark.parametrize("fused_loss", [True, False])
@pytest.mark.parametrize("case", UNALIGNED_CASES)
def test_unaligned_encoder_rows_training_chain(case, fused_loss, monkeypatch):
    """Three training steps through the module on unaligned enc_a / enc_i, on both cuts, against the aligned run.  The forward's scalar
    context loop rounds differently from the float4 one, and the chain carries that into every gradient: measured on a B200, grad_err
    at most 8.2e-6 (v_beta_2.bias of l2size-4cta; 5.8e-6 for the other gradients); checked at 2e-5.  The backward kernels themselves
    are checked bit for bit above."""
    mod, x, _, mask, tgts = _make(case)
    for cut in ("fused", "chunks"):
        monkeypatch.setenv("MMB_DECODER_CUT", cut)
        enc_a = x["enc_a"].clone().requires_grad_(True)
        enc_i = x["enc_i"].clone().requires_grad_(True)
        want_loss, want_h, want_p = _chain(mod, x, mask, tgts, fused_loss, enc_a, enc_i)
        want_p = {n: g.clone() for n, g in want_p.items()}
        ua, ba = _unaligned(x["enc_a"])
        ui, bi = _unaligned(x["enc_i"])
        ba.requires_grad_(True)
        bi.requires_grad_(True)
        ua, ui = ba[1:].view(ua.shape), bi[1:].view(ui.shape)                    # views of the leaves: the gradient lands in ba / bi
        assert ua.data_ptr() % 16 == 4 and ui.data_ptr() % 16 == 4
        loss, d_h, grads = _chain(mod, x, mask, tgts, fused_loss, ua, ui)
        errs = _grad_errs(loss, ba.grad[1:].view(ua.shape), bi.grad[1:].view(ui.shape), d_h, grads,
                          (want_loss, enc_a.grad, enc_i.grad, want_h, want_p))
        bad = {n: e for n, e in errs.items() if e >= 2e-5}
        assert not bad, (cut, bad)


# ---- roll-outs on the paths above ---------------------------------------------------------------------------------------------------

def _greedy_loop(seq, x, mask_u8, steps):
    """The greedy roll-out as a host loop of the step kernel (models.py:184,193: each step's arg-max text row is the next input)."""
    from mmbidaf_b200 import ops
    B = seq.B
    rows = torch.arange(B, device=mask_u8.device)
    sent = x["emb"].new_zeros(B, seq.E)
    h, cell, cov = x["h"], x["h"].new_zeros(B, seq.H), x["h"].new_zeros(B, seq.Lt)
    probs, picks = [], []
    for _ in range(steps):
        p, h, cell, _, cov, am, _, _ = ops.decoder_step_fwd(seq, sent, h, cell, cov, mask_u8, want_argmax=True)
        sent = x["emb"][rows, am].contiguous()
        probs.append(p)
        picks.append(am)
    return torch.stack(probs, 1), torch.stack(picks, 1)


def _oracle_along(mod, x, mask, picks):
    """The oracle in float64 fed the kernel's picks: each step's distribution (B, steps, M)."""
    p = _p64(mod)
    B, steps = picks.shape
    emb = x["emb"].double()
    rows = torch.arange(B, device=emb.device)
    h, cell = x["h"].double().unsqueeze(1), torch.zeros(1, B, mod.hidden_size, dtype=torch.float64, device=emb.device)
    cov = torch.zeros(B, emb.shape[1], 1, dtype=torch.float64, device=emb.device)
    sent = torch.zeros(B, 1, emb.shape[2], dtype=torch.float64, device=emb.device)
    enc_a, enc_i = x["enc_a"].double(), x["enc_i"].double()
    out = []
    for s in range(steps):
        probs, h, cell, _, cov = O.decoder_step(p, sent, h, cell, enc_a, enc_i, cov, mask)
        out.append(probs)
        sent = emb[rows, picks[:, s]].unsqueeze(1)
    return torch.stack(out, 1)


@pytest.mark.parametrize("case", ODD)
def test_odd_hidden_roll_outs_equal_the_host_loop(case, monkeypatch):
    """D = 66 (no stage, scalar loops): the greedy roll-out and the beam roll-out (width 3) of a standalone decoder module bit for bit
    against host loops of the step kernel (a whole model cannot take an odd hidden size: BiDAF wants d % 4 == 0)."""
    from mmbidaf_b200 import ops
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    mod, x, lens, mask, _ = _make(case)
    mod.eval()
    seq = _seq(mod, x["enc_a"], x["enc_i"])
    probs, picks, _ = ops.decoder_greedy_fwd(seq, x["emb"], x["h"], mask.to(torch.uint8), 16)
    want_probs, want_picks = _greedy_loop(seq, x, mask.to(torch.uint8), 16)
    assert torch.equal(picks, want_picks) and torch.equal(probs, want_probs)
    tokens, parents, scores, bprobs, _, _ = mod.beam(x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, lens, 8, 3)
    rt, rp, rs, rprob = _beam_reference(mod, x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, lens, 8, 3)
    assert torch.equal(tokens, rt) and torch.equal(parents, rp) and torch.equal(scores, rs) and torch.equal(bprobs, rprob)


@pytest.mark.parametrize("shape", [(16, 4096), (2, 4096)])
def test_long_lecture_greedy_kernel_equals_the_step_kernel_loop(shape, monkeypatch):
    """The greedy roll-out kernel at long-lecture shapes (L2 by size, 8 CTAs, chunk 512 rows) bit for bit against 16 calls of the
    step kernel (attention.py: MultimodalAttentionDecoder.greedy) -- B * Lt > 20 000 takes the chunk cut by default, so the step kernel
    is forced."""
    from mmbidaf_b200 import ops
    from mmbidaf_b200.layers import MultimodalAttentionDecoder
    B, Lt = shape
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    torch.manual_seed(88 + B)
    mod = MultimodalAttentionDecoder(300, 100, Lt).cuda().eval()
    x = {"enc_a": torch.randn(B, Lt, 200, device="cuda"), "enc_i": torch.randn(B, Lt, 200, device="cuda"),
         "emb": torch.randn(B, Lt, 300, device="cuda"), "h": torch.randn(B, 100, device="cuda")}
    lens = torch.randint(2, Lt + 1, (B,), device="cuda")
    mask_u8 = (torch.arange(Lt, device="cuda").unsqueeze(0) < lens.unsqueeze(1)).to(torch.uint8)
    seq = _seq(mod, x["enc_a"], x["enc_i"])
    probs, picks, _ = ops.decoder_greedy_fwd(seq, x["emb"], x["h"], mask_u8, 16)
    want_probs, want_picks = _greedy_loop(seq, x, mask_u8, 16)
    assert torch.equal(picks, want_picks) and torch.equal(probs, want_probs)


@pytest.mark.parametrize("case", ["long-lecture", "odd-8cta"])
def test_greedy_roll_out_stays_on_the_fp64_oracle(case):
    """The greedy roll-out kernel's 16 distributions against the fp64 oracle fed the kernel's own picks."""
    from mmbidaf_b200 import ops
    mod, x, _, mask, _ = _make(case)
    mod.eval()
    seq = _seq(mod, x["enc_a"], x["enc_i"])
    probs, picks, _ = ops.decoder_greedy_fwd(seq, x["emb"], x["h"], mask.to(torch.uint8), 16)
    want = _oracle_along(mod, x, mask, picks)
    errs = [rel_err(probs[:, s], want[:, s]) for s in range(16)]
    assert max(errs) < TOL, errs
