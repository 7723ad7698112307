"""GPU: the forced roll-out that saves every step (mmb_decoder_forced_train_fused) and the reverse roll-out (mmb_decoder_forced_bwd_fused)
on every launch path of tests/test_rollout_paths_gpu.py: its ROLL_CASES (staged and L2 arms by size and by width, D = 66, 194 and 256,
ranks without text rows, 8- and 4-CTA clusters), unaligned encoder rows and MMB_DEC_STAGE=0 in a child process -- bit for bit against
the host loops of the step kernels (tests/test_sequence_scores_gpu.py), and the gradients against the fp64 oracle.

Both kernels size their clusters by the B N rows as the forced roll-out does (N = 4 here), so the rows of each case take the paths the
module docstring of tests/test_rollout_paths_gpu.py lists for the forced kind; the backward adds 2 H floats of carried state to the
whole-step backward's shared memory, and its arm follows mmb_decoder_step_fused_bwd's rule for the same rows."""
import os
import subprocess
import sys

import pytest
import torch

import test_decoder_paths_gpu as paths
from conftest import grad_err, rel_err
from test_rollout_paths_gpu import ROLL_CASES, _forced_tokens, _make, _steps, _UnalignedRows
from test_decoder_paths_gpu import _unaligned
from test_score_gpu import _random_tokens
from test_sequence_scores_gpu import _check_kernels, _g_terms, _oracle_objective, _seq

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
N = 4


class _Dec:
    """The decoder as _check_kernels asks for it (its sequence over given encoder rows)."""

    def __init__(self, seq):
        self.seq = seq

    def _sequence(self, enc_a, enc_i):
        return {"seq": self.seq}


@pytest.mark.parametrize("case", list(ROLL_CASES))
def test_kernels_equal_the_host_loops_on_every_path(case, monkeypatch):
    """Both kernels on the case's path, N = 4 candidates (one token out of range), against the host loops of the step kernels: every
    saved slice and per-row gradient bit for bit, d_proj within 1e-6 (the N clusters of a video add into the same rows)."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    mod, x, lens, mask = _make(case)
    tokens, _, _ = _forced_tokens(lens, mod.output_size, N, _steps(case))
    _check_kernels(mod, x["emb"], x["h"], x["enc_a"], x["enc_i"], mask, tokens, seed=len(case))


@pytest.mark.parametrize("case", paths.UNALIGNED_CASES)
def test_unaligned_encoder_rows_equal_the_host_loops(case, monkeypatch):
    """enc_a / enc_i at a one-float offset (no row stage, scalar context loop): both kernels against host loops whose step kernels read
    the same unaligned rows, bit for bit."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    mod, x, lens, mask = _make(case)
    ua, _ = _unaligned(x["enc_a"])
    ui, _ = _unaligned(x["enc_i"])
    dec = _UnalignedRows(mod, ua, ui)
    assert dec.seq.enc_a.data_ptr() % 16 == 4
    tokens, _, _ = _forced_tokens(lens, mod.output_size, N, _steps(case))
    _check_kernels(dec, x["emb"], x["h"], ua, ui, mask, tokens, seed=3)


def _kernel_outputs(case):
    """Both kernels' outputs on the case's seeded inputs, on the host: {name: tensor}."""
    from mmbidaf_b200 import ops
    mod, x, lens, mask = _make(case)
    steps = _steps(case)
    tokens, _, _ = _forced_tokens(lens, mod.output_size, N, steps)
    seq = _seq(mod, x["enc_a"], x["enc_i"])
    B, R = lens.shape[0], lens.shape[0] * N
    p_tok, terms, saved = ops.decoder_forced_train_fwd(seq, x["emb"], x["h"].contiguous(), ops._u8(mask), tokens)
    vec_acc, scal_acc = seq.enc_a.new_zeros(R, 6, seq.D), seq.enc_a.new_zeros(R, 4)
    d_proj_a, d_proj_i = torch.zeros_like(seq.proj_a), torch.zeros_like(seq.proj_i)
    grads = ops.decoder_forced_bwd(seq, saved, tokens, _g_terms(steps, R, 7), d_proj_a, d_proj_i, vec_acc, scal_acc)
    names = ("probs", "hw", "alpha", "beta", "ctx12", "pb", "xcat", "gates", "att_cov", "cell", "cov", "h_last")
    out = {"p_tok": p_tok, "terms": terms, **dict(zip(names, saved)), "vec_acc": vec_acc, "scal_acc": scal_acc,
           "d_proj_a": d_proj_a, "d_proj_i": d_proj_i,
           **dict(zip(("d_logits", "d_gates", "d_hw4", "d_ctx12", "d_pre_b", "d_h0"), grads))}
    torch.cuda.synchronize()
    return {name: t.cpu() for name, t in out.items()}


def _stage_child(path, case):
    """Entry point of the child process (MMB_DEC_STAGE=0 in its environment)."""
    torch.save(_kernel_outputs(case), path)


@pytest.mark.parametrize("case", paths.STAGE_CASES)
def test_stage_off_is_bit_identical(case, tmp_path):
    """Both kernels with the row stage (this process) and without it (a child with MMB_DEC_STAGE=0): every output bit for bit but
    d_proj, which the N clusters of a video add in no fixed order (within 1e-6)."""
    if os.environ.get("MMB_DEC_STAGE", "").strip() == "0":
        pytest.skip("MMB_DEC_STAGE=0 in this process: nothing runs staged to compare with")
    off_path = tmp_path / "stage_off.pt"
    env = dict(os.environ, MMB_DEC_STAGE="0", MMB_DECODER_CUT="fused")
    code = ("import sys; sys.path[:0] = sys.argv[1:3]; import test_sequence_scores_paths_gpu as t; "
            "t._stage_child(sys.argv[3], sys.argv[4])")
    args = [sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", code, TESTS, ROOT, str(off_path), case]
    res = subprocess.run(args, env=env, cwd=ROOT, timeout=900, capture_output=True, text=True)
    assert res.returncode == 0, (res.stdout[-2000:], res.stderr[-4000:])
    off = torch.load(off_path, weights_only=True)
    on = _kernel_outputs(case)
    assert set(on) == set(off)
    differ = [name for name in on if not name.startswith("d_proj") and not torch.equal(on[name], off[name])]
    assert not differ, differ
    for name in ("d_proj_a", "d_proj_i"):
        assert rel_err(on[name], off[name]) <= 1e-6, name


ORACLE_CASES = ["long-lecture", "odd-8cta", "d194", "d256", "empty-ranks-8cta", "l2size-4cta"]


@pytest.mark.parametrize("case", ORACLE_CASES)
def test_gradients_stay_on_the_fp64_oracle(case):
    """force_train on the case's path with random per-row weights on logp and loss: the scores within 1e-5 of the fp64 oracle's
    teacher-forced loop, and the gradients of every decoder parameter, enc_a, enc_i and h0 (leaves) within the per-step path's gradient
    tolerances (tests/test_decoder_gpu.py: 5e-5, 5e-4 for the four attention biases whose gradients are cancellation noise, 2e-5 for
    the inputs, each over grad_err's floor)."""
    from mmbidaf_b200.summarize import forced_scores
    mod, x, lens, mask = _make(case)
    steps = _steps(case)
    B = lens.shape[0]
    tokens = _random_tokens(lens.cpu(), N, steps, seed=17)
    g = torch.Generator().manual_seed(len(case))
    w_logp, w_loss = torch.randn(B, N, generator=g).cuda(), torch.randn(B, N, generator=g).cuda()
    leaves = [t.detach().clone().requires_grad_() for t in (x["enc_a"], x["enc_i"], x["h"])]
    mod.zero_grad()
    p_tok, terms = mod.force_train(x["emb"], leaves[2], leaves[0], leaves[1], mask, tokens)
    sc = forced_scores(tokens, p_tok, terms, torch.ones(B, N, dtype=torch.bool, device="cuda"), lens.int())
    ((sc.logp * w_logp).sum() + (sc.loss * w_loss).sum()).backward()
    p = {n: t.detach().double().requires_grad_() for n, t in mod.named_parameters()}
    ref = [t.detach().double().requires_grad_() for t in (x["enc_a"], x["enc_i"], x["h"])]
    obj = _oracle_objective(p, x["emb"].double(), ref[2], ref[0], ref[1], mask, tokens, lens.long(), w_logp.double(), w_loss.double())
    want = ((sc.logp.double() * w_logp).sum() + (sc.loss.double() * w_loss).sum())
    assert rel_err(want, obj) <= 1e-5
    obj.backward()
    for n, t in mod.named_parameters():
        tol = 5e-4 if n in ("v1.bias", "v2.bias", "v_beta_1.bias", "v_beta_2.bias") else 5e-5
        assert grad_err(t.grad, p[n].grad, n) <= tol, n
    for got, w in zip(leaves, ref):
        assert grad_err(got.grad, w.grad) <= 2e-5
