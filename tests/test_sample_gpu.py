"""GPU: sampled summaries -- N roll-outs per video with the pick drawn inside the cluster kernel (mmb_decoder_sample_fused) against a
host loop of the fused step kernel and the standalone pick (mmb_sample_pick), top_k = 1 against greedy, the pick's statistics, the
reproducibility of seeds and of the device key stream, the Summary fields, the shapes of configs 3 and 5, and the errors."""
import copy

import pytest
import torch

from mmbidaf_b200.summarize import _select
from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu


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
        b.text[1, 1:] = 0
        b.text[1, 1] = -1.0
        b.text_len[1] = 2
    return b


def _summarize(model, b, steps, **kw):
    return model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, steps, **kw)


def _decoder_inputs(model, b):
    from mmbidaf_b200.layers.encoding import length_plan
    model.eval()
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    return b.text, h0, enc_a, enc_i, mask, length_plan(b.text_len, b.text.device).len_i32.clone()


def _eligible(mask, eos, used, kept, no_repeat, min_sentences):
    """The constrained rule's eligibility (as tests/test_constrained_gpu.py states it) over (R, M)."""
    idx = torch.arange(mask.shape[-1], device=mask.device)
    avail = eos - (kept if no_repeat else 0)
    eos_ok = ((kept >= min_sentences) | (avail == 0)).unsqueeze(-1)
    below = (idx < eos.unsqueeze(-1)) & ~(used if no_repeat else torch.zeros_like(used))
    return mask & (below | ((idx == eos.unsqueeze(-1)) & eos_ok))


def _sample_reference(dec, emb, h0, enc_a, enc_i, mask, text_len, steps, N, key, T, top_k, no_repeat, min_sentences):
    """The rule as a host loop over B N rows: the fused step kernel on the B-video tensors replicated row-wise (no projection is
    recomputed at B N rows), then mmb_sample_pick, with eligibility tracked as in the constrained greedy reference."""
    from mmbidaf_b200 import _lib, ops
    constrained = no_repeat or min_sentences > 0
    with torch.no_grad():
        seq = dec._sequence(enc_a, enc_i)["seq"]
        B, Lt, H, M = seq.B, seq.Lt, seq.H, seq.M
        R, dev = B * N, emb.device
        rs = copy.copy(seq)
        for f in ("proj_a", "proj_i", "enc_a", "enc_i"):
            setattr(rs, f, getattr(seq, f).repeat_interleave(N, 0).contiguous())
        rs.B, rs.nch = R, _lib.lib().mmb_decoder_chunks(R, Lt)
        rs.counters = torch.zeros(2, R, device=dev, dtype=torch.int32)
        emb_r, mask_r = emb.repeat_interleave(N, 0), mask.bool().repeat_interleave(N, 0)
        eos = text_len.long().repeat_interleave(N) - 1
        base = torch.arange(B, device=dev, dtype=torch.int32).repeat_interleave(N)
        rows = torch.arange(R, device=dev)
        used = torch.zeros(R, M, dtype=torch.bool, device=dev)
        kept = torch.zeros(R, dtype=torch.long, device=dev)
        sent, h = emb.new_zeros(R, emb.shape[2]), h0.reshape(B, H).repeat_interleave(N, 0).contiguous()
        cell, cov = torch.zeros(R, H, device=dev), torch.zeros(R, Lt, device=dev)
        P, picks = [], []
        for s in range(steps):
            p, h, cell, _, cov, *_ = ops.decoder_step_fwd(rs, sent.contiguous(), h, cell, cov, ops._u8(mask_r))
            el = _eligible(mask_r, eos, used, kept, no_repeat, min_sentences) if constrained else None
            pick = ops.sample_pick(p, key, base, steps, s, N, T, top_k, eligible=el)
            pick = torch.where(pick < 0, eos, pick)
            below = pick < eos
            kept = kept + below.long()
            used[rows[below], pick[below]] = True
            sent = emb_r[rows, pick.clamp(0, Lt - 1)]
            P.append(p)
            picks.append(pick)
        return torch.stack(P, 1).view(B, N, steps, M), torch.stack(picks, 1).view(B, N, steps)


def _check(model, b, steps, N, T, top_k, no_repeat, min_sentences, seed=11):
    from mmbidaf_b200 import ops
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    key = ops.seed_key(seed, "cuda")
    probs, tokens = dec.sample(emb, h0, enc_a, enc_i, mask, lens, steps, N, key, T, top_k, no_repeat, min_sentences)
    rp, rt = _sample_reference(dec, emb, h0, enc_a, enc_i, mask, lens, steps, N, key, T, top_k, no_repeat, min_sentences)
    assert torch.equal(tokens, rt)
    assert torch.equal(probs, rp)
    return tokens


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("N", [1, 4])
@pytest.mark.parametrize("T,top_k", [(1.0, 0), (0.7, 3), (1.0, 8), (0.7, 0)])
@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_sample_equals_the_host_loop(tier, B, N, T, top_k, no_repeat, min_sentences):
    tokens = _check(_model(64), _batch(B).to("cuda"), 16, N, T, top_k, no_repeat, min_sentences)
    if no_repeat:
        lens = _batch(B).text_len
        for v in range(B):
            for row in tokens[v].tolist():
                chosen = _select(row, int(lens[v]))
                assert len(set(chosen)) == len(chosen) and len(chosen) >= min(3, int(lens[v]) - 1)


def test_long_lecture_sample_equals_the_host_loop(monkeypatch):
    from mmbidaf_b200 import ops
    model = _model(700)
    b = make_batch(32, 700, 60, 6, 6, seed=41).to("cuda")
    assert ops.decoder_cut(32, 700) == "chunks"            # the sampled roll-out runs the cluster kernel; so must the reference
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    _check(model, b, 6, 2, 1.0, 3, True, 3)
    _check(model, b, 6, 1, 0.7, 0, False, 0)


@pytest.mark.parametrize("B", [1, 3, 21])
@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_top_k_one_is_the_greedy_summary(B, no_repeat, min_sentences):
    model = _model(64)
    b = _batch(B).to("cuda")
    greedy = _summarize(model, b, 16, no_repeat=no_repeat, min_sentences=min_sentences)
    for T, seed in ((1.0, 1), (0.3, 2), (5.0, None)):
        got = _summarize(model, b, 16, num_samples=1, temperature=T, top_k=1, seed=seed, no_repeat=no_repeat,
                         min_sentences=min_sentences)
        assert torch.equal(got.indices, greedy.indices) and torch.equal(got.counts, greedy.counts)
        assert torch.equal(got.out_distributions, greedy.out_distributions)


@pytest.mark.parametrize("T", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("top_k", [0, 3])
@pytest.mark.parametrize("with_eligible", [False, True])
def test_pick_frequencies_follow_p_to_the_one_over_t(T, top_k, with_eligible):
    from scipy.stats import chisquare
    from mmbidaf_b200 import ops
    p = torch.tensor([[0.05, 0.0, 0.3, 0.15, 0.0, 0.25, 0.1, 0.15],
                      [0.5, 0.2, 0.1, 0.1, 0.05, 0.05, 0.0, 0.0]], dtype=torch.float32)
    el = torch.tensor([[1, 1, 1, 0, 1, 1, 1, 1], [1, 0, 1, 1, 1, 1, 1, 0]], dtype=torch.bool)
    R = 20000
    probs = p.repeat(R, 1).cuda()
    eligible = el.repeat(R, 1).cuda() if with_eligible else None
    key = ops.seed_key(1234, "cuda")
    picks = ops.sample_pick(probs, key, torch.arange(2 * R, device="cuda", dtype=torch.int32), 16, 5, 1, T, top_k, eligible)
    picks = picks.view(R, 2).cpu()
    for row in range(2):
        cand = (p[row] > -1) & (el[row] if with_eligible else True)
        w = torch.where(cand, p[row].double() ** (1.0 / T), torch.zeros(8, dtype=torch.float64))
        if top_k:
            order = sorted(range(8), key=lambda m: (-float(p[row, m]), m))
            top = [m for m in order if cand[m]][:top_k]
            w = torch.tensor([float(w[m]) if m in top else 0.0 for m in range(8)], dtype=torch.float64)
        freq = torch.bincount(picks[:, row], minlength=8).double()
        assert (freq[w == 0] == 0).all(), (freq, w)                   # zero-probability and non-candidate sentences never
        nz = w > 0
        expected = w[nz] / w[nz].sum() * R
        assert chisquare(freq[nz].numpy(), expected.numpy()).pvalue > 1e-4


def test_same_seed_same_samples_and_the_key_stream_advances():
    from mmbidaf_b200 import ops
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    b = make_batch(4, 37, 45, 7, 12, seed=3).to("cuda")
    a1 = _summarize(model, b, 12, num_samples=4, seed=7)
    a2 = _summarize(model, b, 12, num_samples=4, seed=7)
    assert torch.equal(a1.samples.tokens, a2.samples.tokens) and torch.equal(a1.samples.probs, a2.samples.probs)
    other = _summarize(model, b, 12, num_samples=4, seed=8)
    assert not torch.equal(a1.samples.tokens, other.samples.tokens)
    summarizer = Summarizer(model)
    for _ in range(2):
        got = summarizer(b, num_samples=4, seed=7)
        assert torch.equal(got.samples.tokens, a1.samples.tokens) and torch.equal(got.indices, a1.indices)
    # seed None: consecutive replays draw fresh keys; after rng_seed the sequence repeats
    summarizer(b, num_samples=4, temperature=2.0)              # capture (the warm-up creates the key state)
    ops.rng_seed(99)
    first = [summarizer(b, num_samples=4, temperature=2.0).samples.tokens.clone() for _ in range(3)]
    assert not torch.equal(first[0], first[1]) and not torch.equal(first[1], first[2])
    ops.rng_seed(99)
    again = [summarizer(b, num_samples=4, temperature=2.0).samples.tokens.clone() for _ in range(3)]
    assert all(torch.equal(x, y) for x, y in zip(first, again))
    assert len(summarizer.buckets) == 2


@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_summary_fields(no_repeat, min_sentences):
    model = _model(64)
    b = _batch(3).to("cuda")
    got = _summarize(model, b, 16, num_samples=8, temperature=1.5, top_k=0, seed=5, no_repeat=no_repeat,
                     min_sentences=min_sentences)
    smp = got.samples
    B, N, S, M = smp.probs.shape
    lens = b.text_len
    want = torch.zeros(B, N, dtype=torch.float64)
    for v in range(B):
        for n in range(N):
            for s in range(S):
                t = int(smp.tokens[v, n, s])
                want[v, n] += torch.log(smp.probs[v, n, s, t].double()).item()
                if t == lens[v] - 1:
                    break
    assert torch.allclose(smp.logp.cpu().double(), want, rtol=1e-6, atol=0)
    best = smp.logp.argmax(1).cpu()
    per = smp.summaries(lens)
    lists = got.to_lists()
    for v in range(B):
        assert lists[v] == per[v][int(best[v])][0]
        assert torch.equal(got.out_distributions[v], smp.probs[v, int(best[v])])
        assert [x[0] for x in per[v]] == [_select(r, int(lens[v])) for r in smp.tokens[v].tolist()]
    assert got.loss is None and got.beams is None


def test_sampled_roll_outs_launch_at_config3_and_config5_shapes():
    from mmbidaf_b200 import ops
    torch.manual_seed(0)
    D, H, E = 200, 100, 300
    for B, Lt in ((32, 409), (16, 4096)):
        model = _model(Lt)
        dec = model.multimodal_att_decoder
        model.eval()
        enc_a, enc_i = torch.randn(B, Lt, D, device="cuda"), torch.randn(B, Lt, D, device="cuda")
        emb, h0 = torch.randn(B, Lt, E, device="cuda"), torch.randn(B, 1, H, device="cuda")
        lens = torch.randint(5, Lt + 1, (B,), device="cuda", dtype=torch.int32)
        eos = lens.view(-1, 1, 1).long() - 1
        mask = torch.arange(Lt, device="cuda").view(1, -1) < lens.view(-1, 1)
        dec.prepare()
        key = ops.seed_key(3, "cuda")
        for top_k, nr, ms in ((0, False, 0), (8, True, 3)):
            probs, tokens = dec.sample(emb, h0, enc_a, enc_i, mask, lens, 4, 4, key, 1.0, top_k, nr, ms)
            assert torch.isfinite(probs).all() and ((tokens >= 0) & (tokens < Lt)).all()
            if ms:
                assert (tokens <= eos).all() and (tokens[:, :, :3] < eos).all()


def test_errors_are_raised_before_any_launch_and_by_the_c_abi():
    from mmbidaf_b200 import _lib, ops
    model = _model(64)
    b = _batch(3).to("cuda")
    before = ops.launch_count
    bad = [dict(num_samples=0), dict(num_samples=65), dict(num_samples=2.0), dict(num_samples=2, temperature=0.0),
           dict(num_samples=2, temperature=float("inf")), dict(num_samples=2, temperature=float("nan")), dict(num_samples=2, top_k=9),
           dict(num_samples=2, top_k=-1), dict(num_samples=2, seed=1.5), dict(num_samples=2, beam_width=2), dict(temperature=0.5),
           dict(top_k=2), dict(seed=3)]
    for kw in bad:
        with pytest.raises(ValueError):
            _summarize(model, b, 4, **kw)
    with pytest.raises(ValueError, match="targets"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, num_samples=2)
    assert ops.launch_count == before
    L = _lib.lib()
    x = torch.zeros(64, device="cuda")
    key = ops.seed_key(1, "cuda")
    t = torch.zeros(64, dtype=torch.int64, device="cuda")
    args = [x.data_ptr()] * 24 + [None, key.data_ptr(), x.data_ptr(), t.data_ptr()]

    def call(B=1, M=4, S=2, N=2, T=1.0, top_k=0, nr=0, ms=0, Lt=4):
        return L.mmb_decoder_sample_fused(*args, B, Lt, 8, 4, 4, M, S, N, T, top_k, nr, ms, _lib.stream())
    for kw in (dict(N=0), dict(N=65), dict(T=0.0), dict(T=-1.0), dict(T=float("inf")), dict(T=float("nan")), dict(top_k=9),
               dict(top_k=-1), dict(nr=2), dict(ms=-1)):
        assert call(**kw) == 1, kw                          # MMB_ERR_INVALID
    assert call(B=1 << 10, M=1 << 12, S=1 << 8, N=64) == 2     # MMB_ERR_UNSUPPORTED: more counters than 2^32
    args[24] = t.data_ptr()                                # (a text_len: the constrained kernel's sentence bits)
    assert call(M=8 * 16384 + 8, S=1, N=1, nr=1) == 2          # MMB_ERR_UNSUPPORTED: more than 16384 sentences per CTA
    assert L.mmb_sample_pick(x.data_ptr(), None, key.data_ptr(), t.data_ptr(), 1, 4, 2, 2, 1, 1.0, 0, t.data_ptr(),
                             _lib.stream()) == 1      # s >= S
    torch.cuda.synchronize()                               # nothing was launched: the device is still usable
    got = _summarize(model, b, 4, num_samples=2, seed=1)
    assert torch.equal(got.indices, _summarize(model, b, 4, num_samples=2, seed=1).indices)


def _hash32(c, k0, k1):
    """common.cuh::hash32 on the host (numpy uint32, wrapping)."""
    import numpy as np
    x = c ^ np.uint32(k0)
    x = x * np.uint32(0x9E3779B1)
    x ^= x >> np.uint32(16)
    x = x * np.uint32(0x85EBCA6B)
    x ^= np.uint32(k1)
    x ^= x >> np.uint32(13)
    x = x * np.uint32(0xC2B2AE35)
    x ^= x >> np.uint32(16)
    return x


@pytest.mark.parametrize("top_k", [0, 2])
def test_the_largest_uniform_gives_a_finite_score(top_k):
    """At the counter whose hash gives the largest uniform (1 - 2^-24), a sentence of probability 1e-30 must still lose to one of
    probability 1, and one of probability 0 must lose too (u = 1 would score them +inf and NaN)."""
    import numpy as np
    from mmbidaf_b200 import ops
    key = ops.seed_key(77, "cuda")
    kv = int(key.item()) & 0xFFFFFFFFFFFFFFFF
    k0, k1 = kv & 0xFFFFFFFF, kv >> 32
    c0, chunk = None, 1 << 24
    for start in range(0, 1 << 30, chunk):
        c = np.arange(start, start + chunk, dtype=np.uint32)
        hit = np.nonzero((_hash32(c, k0, k1) >> np.uint32(9)) == (1 << 23) - 1)[0]
        if len(hit):
            c0 = start + int(hit[0])
            break
    assert c0 is not None
    # M = 2, N = 1, S = 1, s = 0: the counter of sentence m of row r is 2 row_base[r] + m
    hi = c0 & 1
    rows = torch.zeros(2, 2)
    rows[0, hi], rows[0, 1 - hi] = 1e-30, 1.0
    rows[1, hi], rows[1, 1 - hi] = 0.0, 1.0
    base = torch.full((2,), c0 >> 1, dtype=torch.int32, device="cuda")
    for T in (0.5, 1.0, 4.0):
        picks = ops.sample_pick(rows.cuda(), key, base, 1, 0, 1, T, top_k)
        assert picks.tolist() == [1 - hi, 1 - hi]


@pytest.mark.parametrize("top_k", [0, 3])
def test_no_candidate_picks_eos(top_k):
    """A mask that hides the rows below EOS leaves a constrained roll-out no candidate before min_sentences: the pick is EOS."""
    from mmbidaf_b200 import ops
    model = _model(64)
    b = _batch(3).to("cuda")
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    mask = mask.clone()
    mask[0, :int(lens[0]) - 1] = False                    # video 0: every sentence hidden, only its EOS row is left
    mask[2, :(int(lens[2]) - 1) // 2] = False             # video 2: the first half hidden
    dec = model.multimodal_att_decoder
    key = ops.seed_key(5, "cuda")
    probs, tokens = dec.sample(emb, h0, enc_a, enc_i, mask, lens, 16, 4, key, 1.0, top_k, True, 3)
    rp, rt = _sample_reference(dec, emb, h0, enc_a, enc_i, mask, lens, 16, 4, key, 1.0, top_k, True, 3)
    assert torch.equal(tokens, rt) and torch.equal(probs, rp)
    assert (tokens[0] == int(lens[0]) - 1).all()
    assert (tokens[2] >= (int(lens[2]) - 1) // 2).all()


@pytest.mark.parametrize("bad", ["probs_dtype", "probs_dim", "row_base", "key", "eligible_shape", "eligible_dtype", "step"])
def test_sample_pick_checks_its_arguments(bad):
    from mmbidaf_b200 import ops
    probs = torch.zeros(3, 5, device="cuda") if bad != "probs_dtype" else torch.zeros(3, 5, dtype=torch.float64, device="cuda")
    if bad == "probs_dim":
        probs = torch.zeros(15, device="cuda")
    row_base = torch.zeros(3 if bad != "row_base" else 2, dtype=torch.int32, device="cuda")
    key = torch.zeros(1 if bad != "key" else 2, dtype=torch.int64, device="cuda")
    eligible = {"eligible_shape": torch.ones(3, 4, dtype=torch.bool, device="cuda"),
                "eligible_dtype": torch.ones(3, 5, device="cuda")}.get(bad)
    with pytest.raises(ValueError, match="sample_pick"):
        ops.sample_pick(probs, key, row_base, 4, 4 if bad == "step" else 0, eligible=eligible)
    ok = ops.sample_pick(torch.full((3, 5), 0.2, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
                         torch.zeros(3, dtype=torch.int32, device="cuda"), 4, 0, eligible=torch.ones(3, 5, dtype=torch.bool, device="cuda"))
    assert ((ok >= 0) & (ok < 5)).all()
