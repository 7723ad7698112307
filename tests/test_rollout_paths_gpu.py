"""GPU: every summarisation roll-out kernel of csrc/decoder_fused.cu on every launch path of launch_fused, bit for bit against the
host loops of the step kernel that the feature tests use as references, and against the fp64 oracle (oracle.mmbidaf_oracle).

The nine roll-outs: constrained greedy and beam (dec_greedy_constrained_kernel, dec_beam_constrained_kernel), sampled
(dec_sample_kernel, dec_sample_constrained_kernel), nucleus (dec_sample_nucleus_kernel, dec_sample_nucleus_constrained_kernel),
stochastic beam (dec_beam_sample_kernel, dec_beam_sample_constrained_kernel) and forced (dec_forced_kernel); section 2 adds the plain
beam (dec_beam_fused_kernel).  The paths are those of tests/test_decoder_paths_gpu.py, with what a roll-out changes in them:

- Cluster size: 8 CTAs when rows * 8 <= 160, else 4, where rows = B for the greedy and beam kinds and rows = B N for the sampled,
  nucleus and forced roll-outs (one cluster per (video, sample)).  chunk = ceil(Lt / CTAs).
- Shared memory: fused_smem_bytes (the step's base arrays), then the mode's own region behind them -- beam_floats(K) for the beam
  slots (constrained: also every slot's eligible bits), beam_floats(0) for the sampled exchange, nucleus_floats(M) behind that for the
  nucleus row and histogram, beam_floats(K) + kStochBeamExtra + stoch_floats(K) for the stochastic beam.  The row stage (2 chunk D
  floats) goes behind the lot only if the total fits in 232 448 B (227 KB), D % 4 == 0, the row pointers are 16-byte aligned and
  MMB_DEC_STAGE is not 0.

Bytes below are the dynamic shared memory the stage would take the launch to (base arrays + mode region + stage), for the settings
this file runs (N = 4, K = 3); "B / B N" is the cluster size of the roll-outs over B rows / over B N rows.

  case              (B, Lt, hidden, E, M)      CTAs B / B N  chunk      arm           why
  staged-8cta       (3, 24, 100, 300, 409)     8 / 8         3          staged        55 296 (forced) .. 62 560 (constrained stochastic beam)
  config3-4cta      (32, 409, 100, 300, 409)   4 / 4         103        staged        216 496 forced, 218 192 sampled, 222 208 nucleus,
                                                                                      225 008 / 225 168 beam / constrained beam,
                                                                                      227 584 / 227 744 stochastic: all <= 232 448
  l2size-4cta       (32, 600, 100, 300, 600)   4 / 4         150        L2 by size    292 256 .. 305 840 > 232 448
  l2size-8cta       (16, 1250, 100, 300, 1250) 8 / 4         157 / 313  L2 by size    303 552 .. 317 232 (8 CTAs), 555 024 .. 564 096 (4)
  long-lecture      (2, 4096, 100, 300, 4096)  8 / 8         512        L2 by size    875 792 .. 906 624
  empty-ranks       (21, 3, 100, 300, 9)       4 / 4         1          staged        52 080 .. 58 464; rank 3 holds no text rows
  odd-8cta          (5, 37, 33, 10, 40)        8 / 8         5          L2 by width   D = 66: no stage, scalar context loop (20 rows: 8 CTAs)
  odd-4cta          (21, 500, 33, 300, 500)    4 / 4         125        L2 by width   D = 66 on 4-CTA clusters
  d194              (3, 50, 97, 300, 64)       8 / 8         7          L2 by width   D = 194: seven column registers, scalar context loop
  d256              (4, 40, 128, 300, 64)      8 / 8         5          staged        67 936 .. 74 896; D = 256, all eight column registers
  empty-ranks-8cta  (2, 3, 100, 300, 5)        8 / 8         1          staged        52 080 .. 58 176; ranks 3-7 hold no text rows, ranks
                                                                                      5-7 no sentences (ceil(5 / 8) = 1); video 0 has two
                                                                                      sentences below EOS, so min_sentences = 3 reaches
                                                                                      the avail == 0 side of the constrained rule

  config-3 widths (32, 409, 100, 300, 409), 4 CTAs, chunk 103:
    beam, constrained beam       staged up to K = 6 (231 824 / 232 080 B), L2 from K = 7 (234 096 / 234 384)
    stochastic beam, constrained staged up to K = 4 (230 272 / 230 464 B), L2 from K = 5 (232 960 / 233 184)
  rows at staged-8cta: N = 2 -> 6 rows, 8 CTAs, chunk 3; N = 8 -> 24 rows, 4 CTAs, chunk 6 (staged: 61 824 B at most)

Every arm, cluster size and chunk above was confirmed on a B200 by printing them from launch_fused in a build made for that purpose.

The references run the step kernel over the same rows as the roll-out (B rows once per beam slot; B N rows replicated for the
sampled, nucleus and forced kinds), so both sides have the same cluster size and chunk, and the stage arms agree bit for bit
(test_decoder_paths_gpu.test_stage_off_is_bit_identical): every comparison with a host loop is exact.

  L2 by alignment  enc_a / enc_i at a one-float offset: the roll-out and its host loop on the same unaligned rows (test_unaligned_*)
  L2 by switch     MMB_DEC_STAGE=0, read once per process on the first launch, so set in a child process (test_stage_off_*)
"""
import copy
import os
import subprocess
import sys
from unittest import mock

import pytest
import torch

import test_decoder_paths_gpu as paths
from conftest import rel_err
from mmbidaf_b200 import ops
from oracle import mmbidaf_oracle as O
from test_beam_gpu import _reference as _beam_reference
from test_beam_sample_gpu import _reference as _stoch_reference
from test_constrained_gpu import _beam_reference as _cbeam_reference
from test_constrained_gpu import _greedy_reference
from test_decoder_paths_gpu import CASES, _oracle_along, _p64, _unaligned
from test_nucleus_gpu import _reference as _nucleus_reference
from test_sample_gpu import _sample_reference
from test_score_gpu import _forced_reference, _random_tokens

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
TOL = 1e-5

ROLL_CASES = dict(CASES, **{"empty-ranks-8cta": ((2, 3, 100, 300, 5), "staged")})
KERNELS = ("greedy_c", "beam_c", "sample", "sample_c", "nucleus", "nucleus_c", "stoch", "stoch_c", "forced")
N, K = 4, 3                    # samples / candidates per video, beam width
T, TOP_P, SEED = 0.7, 0.8, 11
NO_REPEAT, MIN_SENTENCES = True, 3           # the constrained runs (names ending in _c)
STOCH = ("tokens", "parents", "scores", "probs", "phi", "keys", "paths", "path_slots", "kappa")


def _make(case):
    """test_decoder_paths_gpu._make for the cases here too (empty-ranks-8cta is this file's own)."""
    with mock.patch.dict(paths.CASES, {case: ROLL_CASES[case]}):
        mod, x, lens, mask, _ = paths._make(case)
    mod.eval()
    return mod, x, lens, mask


def _steps(case):
    return 6 if case in ("long-lecture", "l2size-8cta") else 8


def _forced_tokens(lens, M, n, steps, seed=5):
    """(B, n, S) tokens in 0..len-1, but for one out-of-range token M + 7 (p = 0, the next input row clamped to Lt - 1), and the same
    rows for the host loop with M - 1 in its place: a sentence past the video's length (p = 0 by the mask, clamped to the same row),
    which the step kernel can take as a target.  Returns (tokens, reference tokens, index of the out-of-range token)."""
    tokens = _random_tokens(lens.cpu(), n, steps, seed)
    v = int(torch.argmin(lens))
    assert int(lens[v]) < M
    at = (v, n - 1, min(2, steps - 1))
    ref = tokens.clone()
    tokens[at], ref[at] = M + 7, M - 1
    return tokens, ref, at


def _constraints(kernel):
    return (NO_REPEAT, MIN_SENTENCES) if kernel.endswith("_c") else (False, 0)


def _rollouts(mod, x, lens, mask, steps, enc, kernels=KERNELS, n=N, k=K, tokens=None):
    """Each named roll-out on the encoder rows ``enc`` (enc_a, enc_i), as the model calls it: {kernel.table: tensor}."""
    emb, h0, ln = x["emb"], x["h"], lens.int()
    key = ops.seed_key(SEED, "cuda")
    out = {}
    for kern in kernels:
        nr, ms = _constraints(kern)
        if kern == "greedy_c":
            probs, picks, _ = mod.greedy(emb, h0, *enc, mask, steps, text_len=ln, no_repeat=nr, min_sentences=ms)
            tabs = {"probs": probs, "picks": picks}
        elif kern in ("beam", "beam_c"):
            tabs = dict(zip(("tokens", "parents", "scores", "probs"), mod.beam(emb, h0, *enc, mask, ln, steps, k, nr, ms)))
        elif kern in ("sample", "sample_c"):
            tabs = {}
            for top_k in (3, 0):
                probs, picks = mod.sample(emb, h0, *enc, mask, ln, steps, n, key, T, top_k, nr, ms)
                tabs.update({f"k{top_k}.probs": probs, f"k{top_k}.tokens": picks})
        elif kern in ("nucleus", "nucleus_c"):
            probs, picks = mod.sample(emb, h0, *enc, mask, ln, steps, n, key, T, 0, nr, ms, top_p=TOP_P)
            tabs = {"probs": probs, "tokens": picks}
        elif kern in ("stoch", "stoch_c"):
            got = dict(zip(STOCH, mod.beam_sample(emb, h0, *enc, mask, ln, steps, k, key, T, nr, ms)))
            tabs = {name: got[name] for name in STOCH if name != "path_slots"}
        else:
            tabs = dict(zip(("probs", "p_tok", "loss_terms"), mod.force(emb, h0, *enc, mask, tokens, want_probs=True)))
        out.update({f"{kern}.{name}": t for name, t in tabs.items()})
    torch.cuda.synchronize()
    return out


def _references(dec, x, lens, mask, steps, enc, kernels=KERNELS, n=N, k=K, tokens=None):
    """The feature tests' host loops of the step kernel for the same runs, with the same keys as _rollouts."""
    emb, h0, ln = x["emb"], x["h"], lens.int()
    key = ops.seed_key(SEED, "cuda")
    out = {}
    for kern in kernels:
        nr, ms = _constraints(kern)
        if kern == "greedy_c":
            tabs = dict(zip(("probs", "picks"), _greedy_reference(dec, emb, h0, *enc, mask, ln, steps, nr, ms)))
        elif kern == "beam":
            tabs = dict(zip(("tokens", "parents", "scores", "probs"), _beam_reference(dec, emb, h0, *enc, mask, ln, steps, k)))
        elif kern == "beam_c":
            tabs = dict(zip(("tokens", "parents", "scores", "probs"), _cbeam_reference(dec, emb, h0, *enc, mask, ln, steps, k, nr, ms)))
        elif kern in ("sample", "sample_c"):
            tabs = {}
            for top_k in (3, 0):
                probs, picks = _sample_reference(dec, emb, h0, *enc, mask, ln, steps, n, key, T, top_k, nr, ms)
                tabs.update({f"k{top_k}.probs": probs, f"k{top_k}.tokens": picks})
        elif kern in ("nucleus", "nucleus_c"):
            probs, picks, _ = _nucleus_reference(dec, emb, h0, *enc, mask, ln, steps, n, key, T, 0, TOP_P, nr, ms)
            tabs = {"probs": probs, "tokens": picks}
        elif kern in ("stoch", "stoch_c"):
            got = _stoch_reference(dec, emb, h0, *enc, mask, ln, steps, k, key, T, nr, ms)
            tabs = {name: got[name] for name in STOCH if name != "path_slots"}
        else:
            tabs = dict(zip(("probs", "p_tok", "loss_terms"), _forced_reference(dec, emb, h0, *enc, mask, tokens)))
        out.update({f"{kern}.{name}": t for name, t in tabs.items()})
    torch.cuda.synchronize()
    return out


def _assert_equal(got, want):
    assert set(got) == set(want)
    differ = [name for name in want if not torch.equal(got[name], want[name])]
    assert not differ, differ


# ---- 1. every roll-out on every case, bit for bit against its host loop ---------------------------------------------------------

@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("case", list(ROLL_CASES))
def test_roll_out_equals_the_host_loop(case, kernel, monkeypatch):
    """One roll-out kind (N = 4 samples or candidates, beam width 3, T = 0.7, top_k 3 and 0, top_p 0.8, no_repeat with
    min_sentences 3 where constrained) on the case's path against its host loop: every table bit for bit."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")           # the host loops' step kernel is the cluster kernel at every B * Lt
    mod, x, lens, mask = _make(case)
    steps = _steps(case)
    tokens, ref_tokens, at = _forced_tokens(lens, mod.output_size, N, steps)
    enc = (x["enc_a"], x["enc_i"])
    got = _rollouts(mod, x, lens, mask, steps, enc, (kernel,), tokens=tokens)
    _assert_equal(got, _references(mod, x, lens, mask, steps, enc, (kernel,), tokens=ref_tokens))
    if kernel == "forced":
        assert got["forced.p_tok"][at] == 0


@pytest.mark.parametrize("n", [2, 8])
def test_rows_set_the_cluster_size(n, monkeypatch):
    """The sampled, nucleus and forced roll-outs size their clusters by B N: at staged-8cta, N = 2 gives 6 rows on 8-CTA clusters
    and N = 8 gives 24 rows on 4-CTA clusters; each equals its host loop bit for bit."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    mod, x, lens, mask = _make("staged-8cta")
    tokens, ref_tokens, _ = _forced_tokens(lens, mod.output_size, n, 8)
    kernels = ("sample", "sample_c", "nucleus", "nucleus_c", "forced")
    enc = (x["enc_a"], x["enc_i"])
    got = _rollouts(mod, x, lens, mask, 8, enc, kernels, n=n, tokens=tokens)
    _assert_equal(got, _references(mod, x, lens, mask, 8, enc, kernels, n=n, tokens=ref_tokens))


# ---- 2. both arms at config-3 shapes ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("k", range(1, 9))
def test_config3_widths_equal_the_host_loop(k, monkeypatch):
    """The beam, constrained beam, stochastic beam and constrained stochastic beam at config-3 shapes (B = 32, Lt = M = 409) and width
    k, 12 steps, against their host loops bit for bit: the row stage is on up to k = 6 for the beams and k = 4 for the stochastic
    beams, and the rows come from L2 above (the module docstring)."""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    mod, x, lens, mask = _make("config3-4cta")
    kernels = ("beam", "beam_c", "stoch", "stoch_c")
    enc = (x["enc_a"], x["enc_i"])
    got = _rollouts(mod, x, lens, mask, 12, enc, kernels, k=k)
    _assert_equal(got, _references(mod, x, lens, mask, 12, enc, kernels, k=k))


# ---- 3. MMB_DEC_STAGE=0 in a child process ----------------------------------------------------------------------------------------

def _stage_outputs(case):
    """Every roll-out of section 1 on the case's seeded inputs; at config 3 also the beams at width 6 and the stochastic beams at
    width 4, the widest widths that run staged there."""
    mod, x, lens, mask = _make(case)
    steps = _steps(case)
    tokens, _, _ = _forced_tokens(lens, mod.output_size, N, steps)
    enc = (x["enc_a"], x["enc_i"])
    out = _rollouts(mod, x, lens, mask, steps, enc, tokens=tokens)
    if case == "config3-4cta":
        for k, kernels in ((6, ("beam", "beam_c")), (4, ("stoch", "stoch_c"))):
            out.update({f"K{k}.{name}": t for name, t in _rollouts(mod, x, lens, mask, steps, enc, kernels, k=k).items()})
    return {name: t.cpu() for name, t in out.items()}


def _stage_child(path, case):
    """Entry point of the child process (MMB_DEC_STAGE=0 in its environment)."""
    torch.save(_stage_outputs(case), path)


@pytest.mark.parametrize("case", paths.STAGE_CASES)
def test_stage_off_is_bit_identical(case, tmp_path):
    """Every roll-out with the row stage (this process) and without it (a child with MMB_DEC_STAGE=0): bit for bit, for the reasons
    test_decoder_paths_gpu.test_stage_off_is_bit_identical gives for the step (D = 200 here)."""
    if os.environ.get("MMB_DEC_STAGE", "").strip() == "0":
        pytest.skip("MMB_DEC_STAGE=0 in this process: nothing runs staged to compare with")
    off_path = tmp_path / "stage_off.pt"
    env = dict(os.environ, MMB_DEC_STAGE="0", MMB_DECODER_CUT="fused")
    code = ("import sys; sys.path[:0] = sys.argv[1:3]; import test_rollout_paths_gpu as t; t._stage_child(sys.argv[3], sys.argv[4])")
    args = [sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", code, TESTS, ROOT, str(off_path), case]
    res = subprocess.run(args, env=env, cwd=ROOT, timeout=900, capture_output=True, text=True)
    assert res.returncode == 0, (res.stdout[-2000:], res.stderr[-4000:])
    off = torch.load(off_path, weights_only=True)
    _assert_equal(_stage_outputs(case), off)


# ---- 4. unaligned enc_a / enc_i ---------------------------------------------------------------------------------------------------

class _UnalignedSeq(ops.DecoderSeq):
    """A sequence whose enc_a / enc_i stay at a 4-byte offset when a host loop replicates them over B N rows (a fresh tensor is
    16-byte aligned), so that the loop's step kernel takes the scalar context loop as the roll-out does."""

    def __setattr__(self, name, value):
        if name in ("enc_a", "enc_i") and value.data_ptr() % 16 == 0:
            value = _unaligned(value)[0]
        super().__setattr__(name, value)


class _UnalignedRows:
    """The decoder as the host loops see it (they only ask it for the sequence) over unaligned encoder rows."""

    def __init__(self, mod, enc_a, enc_i):
        with torch.no_grad():
            self.seq = copy.copy(mod._sequence(enc_a, enc_i)["seq"])
        self.seq.__class__ = _UnalignedSeq

    def _sequence(self, enc_a, enc_i):
        return {"seq": self.seq}


@pytest.mark.parametrize("case", paths.UNALIGNED_CASES)
def test_unaligned_encoder_rows_equal_the_host_loop(case, monkeypatch):
    """Every roll-out on enc_a / enc_i at a one-float offset (L2, scalar context loop) against its host loop on the same unaligned
    rows: bit for bit.  The forced roll-out's tables also lie within 1e-6 of its run on the aligned rows: its picks are given, so only
    the context sums' order differs.  (A sampled pick may legitimately flip on a near tie between the two runs: not compared.)"""
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    mod, x, lens, mask = _make(case)
    steps = _steps(case)
    ua, _ = _unaligned(x["enc_a"])
    ui, _ = _unaligned(x["enc_i"])
    tokens, ref_tokens, _ = _forced_tokens(lens, mod.output_size, N, steps)
    got = _rollouts(mod, x, lens, mask, steps, (ua, ui), tokens=tokens)
    dec = _UnalignedRows(mod, ua, ui)
    assert dec.seq.enc_a.data_ptr() % 16 == 4
    _assert_equal(got, _references(dec, x, lens, mask, steps, (ua, ui), tokens=ref_tokens))
    aligned = _rollouts(mod, x, lens, mask, steps, (x["enc_a"], x["enc_i"]), ("forced",), tokens=tokens)
    errs = {name: rel_err(got[name], t) for name, t in aligned.items()}
    assert max(errs.values()) < 1e-6, errs


# ---- 5. the fp64 oracle along each row's picks ------------------------------------------------------------------------------------

ORACLE_CASES = ["long-lecture", "odd-8cta", "d194", "d256", "empty-ranks-8cta"]


def _replicated(x, mask, n):
    return {name: x[name].repeat_interleave(n, 0) for name in ("enc_a", "enc_i", "emb", "h")}, mask.repeat_interleave(n, 0)


def _check_distributions(got, want, mask, what):
    """got (R, S, M) fp32 against want (R, S, M) fp64: every step within TOL, nothing past a video's length, each row summing to 1."""
    errs = [rel_err(got[:, s], want[:, s]) for s in range(got.shape[1])]
    assert max(errs) < TOL, (what, errs)
    assert (got.masked_select(~mask.unsqueeze(1).expand_as(got)) == 0).all(), what
    assert float((got.double().sum(2) - 1).abs().max()) < 1e-5, what


def _oracle_forced(mod, x, mask, tokens):
    """O.decoder_step in float64 along given token rows (R, S), the next input the clamped row: (probs (R, S, M), coverage terms
    (S, R) = sum_t min(att_cov, coverage'))."""
    p = _p64(mod)
    R, steps = tokens.shape
    emb = x["emb"].double()
    rows = torch.arange(R, device=emb.device)
    h, cell = x["h"].double().unsqueeze(1), torch.zeros(1, R, mod.hidden_size, dtype=torch.float64, device=emb.device)
    cov = torch.zeros(R, emb.shape[1], 1, dtype=torch.float64, device=emb.device)
    sent = torch.zeros(R, 1, emb.shape[2], dtype=torch.float64, device=emb.device)
    enc_a, enc_i = x["enc_a"].double(), x["enc_i"].double()
    probs, terms = [], []
    for s in range(steps):
        pr, h, cell, att, cov = O.decoder_step(p, sent, h, cell, enc_a, enc_i, cov, mask)
        probs.append(pr)
        terms.append(torch.minimum(att, cov).sum(dim=(1, 2)))
        sent = emb[rows, tokens[:, s].clamp(0, emb.shape[1] - 1)].unsqueeze(1)
    return torch.stack(probs, 1), torch.stack(terms)


@pytest.mark.parametrize("case", ORACLE_CASES)
def test_sampled_and_forced_rows_stay_on_the_fp64_oracle(case):
    """Each row of the sampled, nucleus and forced roll-outs (plain and constrained) against the oracle in float64 fed that row's
    picks with its video replicated: every step's distribution within 1e-5, no mass past the video's length, each summing to 1; the
    forced rows' p of their token and both loss terms (-log(p + 1e-12) and the coverage term) within 1e-5."""
    mod, x, lens, mask = _make(case)
    steps = _steps(case)
    M = mod.output_size
    tokens, _, at = _forced_tokens(lens, M, N, steps)
    got = _rollouts(mod, x, lens, mask, steps, (x["enc_a"], x["enc_i"]), ("sample", "sample_c", "nucleus", "nucleus_c", "forced"),
                    tokens=tokens)
    B = lens.shape[0]
    xr, mr = _replicated(x, mask, N)
    for run in ("sample.k3", "sample.k0", "sample_c.k3", "sample_c.k0", "nucleus", "nucleus_c"):
        picks = got[f"{run}.tokens"].reshape(B * N, steps)
        want = _oracle_along(mod, xr, mr, picks)
        _check_distributions(got[f"{run}.probs"].reshape(B * N, steps, M), want, mr, run)
    rows = tokens.reshape(B * N, steps)
    want, want_cov = _oracle_forced(mod, xr, mr, rows)
    _check_distributions(got["forced.probs"].reshape(B * N, steps, M), want, mr, "forced")
    inside = (rows >= 0) & (rows < M)
    want_p = torch.where(inside, want.gather(2, rows.clamp(0, M - 1).unsqueeze(2)).squeeze(2), 0.0)
    assert not inside.all() and got["forced.p_tok"][at] == 0
    terms = got["forced.loss_terms"]
    errs = {"p_tok": rel_err(got["forced.p_tok"].reshape(B * N, steps), want_p),
            "nll": rel_err(terms[:, 0], -torch.log(want_p + 1e-12).t()), "coverage": rel_err(terms[:, 1], want_cov)}
    assert max(errs.values()) < TOL, errs
