"""GPU: nucleus (top-p) summaries -- the draw limited to the nucleus inside the sampled roll-out kernel
(mmb_decoder_sample_nucleus_fused) against a host loop of the fused step kernel and the row reference (mmb_sample_pick_nucleus),
ties across the ranks of a cluster, top_p = 1 against the sampled roll-out and a tiny top_p against greedy, membership and
frequencies of the picks, Summarizer buckets and seeds, the shapes of configs 3 and 5, and the errors."""
import copy

import pytest
import torch

from mmbidaf_b200.decode import nucleus
from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu


def _model(m, seed=224, out_scale=None):
    from mmbidaf_b200.models import MMBiDAF
    params = O.make_params(100, 300, 128, 1000, m, seed=seed)
    model = MMBiDAF(100, 300, 128, 1000, torch.device("cuda"), drop_prob=0.0, max_transcript_length=m)
    model.load_state_dict(params)
    if out_scale is not None:                              # 0: uniform rows over the unmasked sentences; large: peaked rows
        with torch.no_grad():
            model.multimodal_att_decoder.out.weight.mul_(out_scale)
            model.multimodal_att_decoder.out.bias.mul_(out_scale)
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
    """The constrained rule's eligibility over (R, M)."""
    idx = torch.arange(mask.shape[-1], device=mask.device)
    avail = eos - (kept if no_repeat else 0)
    eos_ok = ((kept >= min_sentences) | (avail == 0)).unsqueeze(-1)
    below = (idx < eos.unsqueeze(-1)) & ~(used if no_repeat else torch.zeros_like(used))
    return mask & (below | ((idx == eos.unsqueeze(-1)) & eos_ok))


def _reference(dec, emb, h0, enc_a, enc_i, mask, text_len, steps, N, key, T, top_k, top_p, no_repeat, min_sentences):
    """The rule as a host loop over B N rows: the fused step kernel on the B-video tensors replicated row-wise, then
    mmb_sample_pick_nucleus.  Returns (probs (B,N,S,M), picks (B,N,S), eligible (B,N,S,M) or None)."""
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
        P, picks, els = [], [], []
        for s in range(steps):
            p, h, cell, _, cov, *_ = ops.decoder_step_fwd(rs, sent.contiguous(), h, cell, cov, ops._u8(mask_r))
            el = _eligible(mask_r, eos, used, kept, no_repeat, min_sentences) if constrained else None
            pick = ops.sample_pick(p, key, base, steps, s, N, T, top_k, eligible=el, top_p=top_p)
            pick = torch.where(pick < 0, eos, pick)
            below = pick < eos
            kept = kept + below.long()
            used[rows[below], pick[below]] = True
            sent = emb_r[rows, pick.clamp(0, Lt - 1)]
            P.append(p)
            picks.append(pick)
            els.append(el)
        el = torch.stack(els, 1).view(B, N, steps, M) if constrained else None
        return torch.stack(P, 1).view(B, N, steps, M), torch.stack(picks, 1).view(B, N, steps), el


def _check(model, b, steps, N, T, top_k, top_p, no_repeat, min_sentences, seed=11, membership=False):
    from mmbidaf_b200 import ops
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    dec = model.multimodal_att_decoder
    key = ops.seed_key(seed, "cuda")
    probs, tokens = dec.sample(emb, h0, enc_a, enc_i, mask, lens, steps, N, key, T, top_k, no_repeat, min_sentences, top_p=top_p)
    rp, rt, el = _reference(dec, emb, h0, enc_a, enc_i, mask, lens, steps, N, key, T, top_k, top_p, no_repeat, min_sentences)
    assert torch.equal(probs, rp)
    assert torch.equal(tokens, rt)
    if membership:                                         # every pick lies in the nucleus the host cuts from the returned probs
        pc, tc = probs.cpu(), tokens.cpu()
        ec = el.cpu() if el is not None else None
        sizes = []
        for v in range(pc.shape[0]):
            for n in range(N):
                for s in range(steps):
                    members = nucleus(pc[v, n, s], None if ec is None else ec[v, n, s], top_k, top_p)
                    assert int(tc[v, n, s]) in members or (not members and int(tc[v, n, s]) == int(lens[v]) - 1)
                    sizes.append(len(members))
        return tokens, sizes
    return tokens, None


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 3, 21, 32])
@pytest.mark.parametrize("N", [1, 4])
@pytest.mark.parametrize("top_p", [0.3, 0.9])
@pytest.mark.parametrize("T,top_k", [(1.0, 0), (0.7, 3), (0.7, 0)])
@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_nucleus_equals_the_host_loop(tier, B, N, top_p, T, top_k, no_repeat, min_sentences):
    tokens, _ = _check(_model(64), _batch(B).to("cuda"), 16, N, T, top_k, top_p, no_repeat, min_sentences)
    if no_repeat:
        from mmbidaf_b200.summarize import _select
        lens = _batch(B).text_len
        for v in range(B):
            for row in tokens[v].tolist():
                chosen = _select(row, int(lens[v]))
                assert len(set(chosen)) == len(chosen) and len(chosen) >= min(3, int(lens[v]) - 1)


def test_long_lecture_nucleus_equals_the_host_loop(monkeypatch):
    from mmbidaf_b200 import ops
    model = _model(700)
    b = make_batch(32, 700, 60, 6, 6, seed=41).to("cuda")
    assert ops.decoder_cut(32, 700) == "chunks"            # the sampled roll-out runs the cluster kernel; so must the reference
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    _check(model, b, 6, 2, 1.0, 3, 0.9, True, 3)
    _check(model, b, 6, 1, 0.7, 0, 0.5, False, 0)
    _check(model, b, 6, 2, 1.3, 0, 0.95, True, 2)


@pytest.mark.parametrize("B,N", [(1, 4), (3, 2), (32, 1)])
@pytest.mark.parametrize("top_p", [0.1, 0.5, 0.9])
@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_ties_across_ranks_of_uniform_rows(B, N, top_p, no_repeat, min_sentences):
    """A zeroed output layer gives every step a uniform row over the unmasked sentences: the nucleus ends inside a run of ties that
    spans the ranks of the cluster (B = 1, 3: eight ranks; B = 32: four).  Every pick lies in the host's nucleus of the returned row
    and the roll-out equals the host loop."""
    model = _model(64, out_scale=0.0)
    b = _batch(B).to("cuda")
    _, sizes = _check(model, b, 16, N, 1.0, 0, top_p, no_repeat, min_sentences, membership=True)
    if top_p >= 0.5:
        assert max(sizes) > 8                              # the cut fell inside long runs of ties
    _check(model, b, 16, N, 0.7, 3, top_p, no_repeat, min_sentences, membership=True)


@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_peaked_rows(no_repeat, min_sentences):
    """Large output weights give peaked rows: the nucleus is one sentence on most steps (on fewer under no_repeat, which takes the
    peaks away once they are used)."""
    model = _model(64, out_scale=40.0)
    b = _batch(3).to("cuda")
    _, sizes = _check(model, b, 16, 4, 1.0, 0, 0.9, no_repeat, min_sentences, membership=True)
    assert sum(s == 1 for s in sizes) > len(sizes) // (4 if no_repeat else 2)


@pytest.mark.parametrize("B", [1, 21])
@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_top_p_one_is_the_sampled_roll_out_and_a_tiny_top_p_is_greedy(B, no_repeat, min_sentences):
    model = _model(64)
    b = _batch(B).to("cuda")
    for T, top_k in ((1.0, 0), (0.6, 3)):
        want = _summarize(model, b, 16, num_samples=4, temperature=T, top_k=top_k, seed=9, no_repeat=no_repeat,
                          min_sentences=min_sentences)
        got = _summarize(model, b, 16, num_samples=4, temperature=T, top_k=top_k, seed=9, no_repeat=no_repeat,
                         min_sentences=min_sentences, top_p=1.0)
        assert torch.equal(got.samples.tokens, want.samples.tokens) and torch.equal(got.samples.probs, want.samples.probs)
    greedy = _summarize(model, b, 16, no_repeat=no_repeat, min_sentences=min_sentences)
    for T, top_k, seed in ((1.0, 0, 1), (0.3, 0, 2), (5.0, 0, None), (2.0, 5, None), (0.7, 8, 3)):
        got = _summarize(model, b, 16, num_samples=2, temperature=T, top_k=top_k, seed=seed, no_repeat=no_repeat,
                         min_sentences=min_sentences, top_p=1e-6)
        assert torch.equal(got.indices, greedy.indices) and torch.equal(got.counts, greedy.counts)
        assert torch.equal(got.out_distributions, greedy.out_distributions)


ROWS = [[0.05, 0.0, 0.3, 0.15, 0.0, 0.25, 0.1, 0.15],
        [0.5, 0.2, 0.1, 0.1, 0.05, 0.05, 0.0, 0.0],
        [0.125] * 8]
ELIGIBLE = [[1, 1, 1, 0, 1, 1, 1, 1], [1, 0, 1, 1, 1, 1, 1, 0], [0, 1, 1, 1, 1, 1, 1, 1]]


@pytest.mark.parametrize("T", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("top_k,top_p", [(0, 0.5), (0, 0.8), (3, 0.7), (0, 0.95)])
@pytest.mark.parametrize("with_eligible", [False, True])
def test_picks_hit_the_nucleus_with_frequencies_of_p_to_the_one_over_t(T, top_k, top_p, with_eligible):
    from scipy.stats import chisquare
    from mmbidaf_b200 import ops
    p = torch.tensor(ROWS, dtype=torch.float32)
    el = torch.tensor(ELIGIBLE, dtype=torch.bool)
    R, W = 20000, len(ROWS)
    probs = p.repeat(R, 1).cuda()
    eligible = el.repeat(R, 1).cuda() if with_eligible else None
    key = ops.seed_key(4321, "cuda")
    picks = ops.sample_pick(probs, key, torch.arange(W * R, device="cuda", dtype=torch.int32), 16, 5, 1, T, top_k, eligible, top_p)
    picks = picks.view(R, W).cpu()
    for row in range(W):
        members = nucleus(p[row], el[row] if with_eligible else None, top_k, top_p)
        freq = torch.bincount(picks[:, row], minlength=8).double()
        assert set(torch.nonzero(freq).flatten().tolist()) == set(members), (row, freq, members)   # exactly the nucleus
        w = torch.zeros(8, dtype=torch.float64)
        for m in members:
            w[m] = float(p[row, m]) ** (1.0 / T)
        if len(members) > 1:
            expected = w[members] / w[members].sum() * R
            assert chisquare(freq[members].numpy(), expected.numpy()).pvalue > 1e-4


def test_the_row_reference_picks_inside_the_host_nucleus():
    """Wide rows -- uniform, random, a few distinct values after zeros, very peaked with many q = 0 -- with and without top_k: every
    pick of the row reference (what the host loop tests rest on) lies in the nucleus decode.nucleus cuts."""
    from mmbidaf_b200 import ops
    key = ops.seed_key(8, "cuda")
    M = 300
    rows = torch.full((6, M), 1.0 / M)
    rows[3] = torch.softmax(torch.randn(M, generator=torch.Generator().manual_seed(1)) * 3, 0)
    rows[4, :] = 0.0
    rows[4, :7] = torch.tensor([0.3, 0.2, 0.2, 0.1, 0.1, 0.05, 0.05])
    rows[5] = torch.softmax(torch.randn(M, generator=torch.Generator().manual_seed(2)) * 30, 0)
    base = torch.arange(6, device="cuda", dtype=torch.int32)
    for top_p in (0.2, 0.6, 0.99):
        for top_k in (0, 4):
            picks = ops.sample_pick(rows.cuda(), key, base, 3, 1, 1, 1.0, top_k, top_p=top_p).cpu()
            for r in range(6):
                assert int(picks[r]) in nucleus(rows[r], None, top_k, top_p)


def test_summarizer_seeds_and_buckets():
    from mmbidaf_b200 import ops
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    b = make_batch(4, 37, 45, 7, 12, seed=3).to("cuda")
    eager = _summarize(model, b, 12, num_samples=4, seed=7, top_p=0.8)
    summarizer = Summarizer(model)
    for _ in range(2):
        got = summarizer(b, num_samples=4, seed=7, top_p=0.8)
        assert torch.equal(got.samples.tokens, eager.samples.tokens) and torch.equal(got.indices, eager.indices)
        assert torch.equal(got.samples.probs, eager.samples.probs)
    summarizer(b, num_samples=4, temperature=2.0, top_p=0.95)         # capture (the warm-up creates the key state)
    ops.rng_seed(99)
    first = [summarizer(b, num_samples=4, temperature=2.0, top_p=0.95).samples.tokens.clone() for _ in range(3)]
    assert not torch.equal(first[0], first[1]) and not torch.equal(first[1], first[2])
    ops.rng_seed(99)
    again = [summarizer(b, num_samples=4, temperature=2.0, top_p=0.95).samples.tokens.clone() for _ in range(3)]
    assert all(torch.equal(x, y) for x, y in zip(first, again))
    summarizer(b, num_samples=4, seed=7, top_p=0.5)
    summarizer(b, num_samples=4, seed=7)
    assert len(summarizer.buckets) == 4                                # one per top_p (1.0 included)


def test_nucleus_roll_outs_launch_at_config3_and_config5_shapes():
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
        for top_k, top_p, nr, ms in ((0, 0.9, False, 0), (0, 0.5, True, 3), (8, 0.9, True, 3)):
            probs, tokens = dec.sample(emb, h0, enc_a, enc_i, mask, lens, 4, 4, key, 1.0, top_k, nr, ms, top_p=top_p)
            assert torch.isfinite(probs).all() and ((tokens >= 0) & (tokens < Lt)).all()
            pc, tc, mc = probs[:2].cpu(), tokens[:2].cpu(), mask[:2].cpu()
            for v in range(2):
                e = int(lens[v]) - 1
                for n in range(4):
                    used, kept = torch.zeros(Lt, dtype=torch.bool), 0          # the constrained rule's state, rebuilt from the picks
                    for s in range(4):
                        el = None
                        if ms:
                            el = _eligible(mc[v:v + 1], torch.tensor([e]), used[None], torch.tensor([kept]), nr, ms)[0]
                        assert int(tc[v, n, s]) in nucleus(pc[v, n, s], el, top_k, top_p)
                        t = int(tc[v, n, s])
                        if t < e:
                            kept += 1
                            used[t] = True
            if ms:
                assert (tokens <= eos).all() and (tokens[:, :, :3] < eos).all()


def test_errors_are_raised_before_any_launch_and_by_the_c_abi():
    from mmbidaf_b200 import _lib, ops
    model = _model(64)
    b = _batch(3).to("cuda")
    before = ops.launch_count
    for kw in (dict(num_samples=2, top_p=0.0), dict(num_samples=2, top_p=1.5), dict(num_samples=2, top_p=float("nan")),
               dict(num_samples=2, top_p=True), dict(top_p=0.9), dict(top_p=0.9, beam_width=2)):
        with pytest.raises(ValueError, match="top_p"):
            _summarize(model, b, 4, **kw)
    with pytest.raises(ValueError, match="top_p"):
        model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 4, targets=b.targets, top_p=0.5)
    assert ops.launch_count == before
    L = _lib.lib()
    x = torch.zeros(64, device="cuda")
    key = ops.seed_key(1, "cuda")
    t = torch.zeros(64, dtype=torch.int64, device="cuda")
    args = [x.data_ptr()] * 24 + [None, key.data_ptr(), x.data_ptr(), t.data_ptr()]

    def call(B=1, M=4, S=2, N=2, T=1.0, top_k=0, nr=0, ms=0, Lt=4, top_p=0.5):
        return L.mmb_decoder_sample_nucleus_fused(*args, B, Lt, 8, 4, 4, M, S, N, T, top_k, nr, ms, top_p, _lib.stream())
    for kw in (dict(top_p=0.0), dict(top_p=-0.5), dict(top_p=1.0001), dict(top_p=float("nan")), dict(top_p=float("inf")),
               dict(N=0), dict(T=0.0), dict(top_k=9), dict(nr=2), dict(ms=-1)):
        assert call(**kw) == 1, kw                          # MMB_ERR_INVALID
    assert call(M=65536, S=1, N=1) == 2                     # MMB_ERR_UNSUPPORTED: P Q would not fit 64 bits
    assert call(B=1 << 10, M=1 << 12, S=1 << 8, N=64) == 2
    pick = lambda top_p, M=4: L.mmb_sample_pick_nucleus(x.data_ptr(), None, key.data_ptr(), t.data_ptr(), 1, M, 2, 0, 1, 1.0, 0,
                                                        t.data_ptr(), top_p, _lib.stream())
    assert pick(0.0) == 1 and pick(2.0) == 1 and pick(float("nan")) == 1
    assert pick(0.5, M=65536) == 2
    torch.cuda.synchronize()                               # nothing was launched: the device is still usable
    got = _summarize(model, b, 4, num_samples=2, seed=1, top_p=0.5)
    assert torch.equal(got.indices, _summarize(model, b, 4, num_samples=2, seed=1, top_p=0.5).indices)
