"""GPU: samples without replacement -- the stochastic beam roll-out as one cluster kernel (mmb_decoder_beam_sample_fused) against a
host loop of the fused step kernel that applies the same rule, distinct and constrained samples, the complete enumeration of a tiny
video, the sampling distribution and the unbiased estimate, width 1 against num_samples=1, and graph replay (Summarizer)."""
import math

import numpy as np
import pytest
import torch

from mmbidaf_b200.summarize import Inclusion, _select
from mmbidaf_b200.synth import make_batch
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu

EMPTY, LIVE, DONE = 0, 1, 2
NEG_LN2 = -0.6931471824645996                              # fp32(-ln 2), as the kernel's constant


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


def _short(b, v, n):
    """Video v of batch b as a transcript of n rows (n - 1 sentences and the EOS row)."""
    b.text[v, n - 1:] = 0
    b.text[v, n - 1] = -1.0
    b.text_len[v] = n
    return b


def _batch(B, lt=37, la=45, li=7, t_dec=16, seed=5):
    b = make_batch(B, lt, la, li, t_dec, seed=seed + B)
    return _short(b, 1, 2) if B > 1 else b                 # a two-row transcript: one sentence and the EOS row


def _decoder_inputs(model, b):
    from mmbidaf_b200.layers.encoding import length_plan
    model.eval()
    dec = model.multimodal_att_decoder
    with torch.no_grad():
        enc_a, enc_i, h0, mask = model._encode(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, dec.prepare)
    return b.text, h0, enc_a, enc_i, mask, length_plan(b.text_len, b.text.device).len_i32.clone()


def _hash32(c, k0, k1):
    """common.cuh::hash32 on the host (numpy uint32, wrapping)."""
    x = c ^ np.uint32(k0)
    x = x * np.uint32(0x9E3779B1)
    x ^= x >> np.uint32(16)
    x = x * np.uint32(0x85EBCA6B)
    x ^= np.uint32(k1)
    x ^= x >> np.uint32(13)
    x = x * np.uint32(0xC2B2AE35)
    x ^= x >> np.uint32(16)
    return x


def _uniforms(key, B, S, s, K, M):
    """u (B, K, M) of step s: the sampled rule's uniform of the counter ((b S + s) K + k) M + m."""
    kv = int(key.item()) & 0xFFFFFFFFFFFFFFFF
    b = np.arange(B, dtype=np.uint64).reshape(B, 1, 1)
    k = np.arange(K, dtype=np.uint64).reshape(1, K, 1)
    m = np.arange(M, dtype=np.uint64).reshape(1, 1, M)
    c = ((((b * S + s) * K + k) * M + m) & 0xFFFFFFFF).astype(np.uint32)
    h = _hash32(c, kv & 0xFFFFFFFF, kv >> 32)
    return torch.from_numpy(((h >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23))


def _eligible(mask, eos, used, kept, no_repeat, min_sentences):
    """The constrained rule's eligibility over (..., M) (as tests/test_constrained_gpu.py states it)."""
    idx = torch.arange(mask.shape[-1], device=mask.device)
    e = eos.unsqueeze(-1)
    avail = eos - (kept if no_repeat else 0)
    eos_ok = ((kept >= min_sentences) | (avail == 0)).unsqueeze(-1)
    below = (idx < e) & ~(used if no_repeat else torch.zeros_like(used))
    return mask & (below | ((idx == e) & eos_ok))


def _reference(dec, emb, h0, enc_a, enc_i, mask, text_len, steps, K, key, T, no_repeat, min_sentences):
    """The rule as a host loop: per step the fused step kernel once per slot on all B videos, then the normaliser, the perturbation,
    the truncated keys and the ranking in torch ops on the device (u from the host hash), the state gathered by parent."""
    from mmbidaf_b200 import ops
    with torch.no_grad():
        seq = dec._sequence(enc_a, enc_i)["seq"]
        B, Lt, H, M = seq.B, seq.Lt, seq.H, seq.M
        dev = emb.device
        mask_u8 = ops._u8(mask)
        rows = torch.arange(B, device=dev)
        eos = text_len.long() - 1
        inv = float(np.float32(1.0) / np.float32(T))
        ninf = torch.tensor(-math.inf, device=dev)
        h = torch.zeros(B, K, H, device=dev)
        h[:, 0] = h0.reshape(B, H)
        cell, cov = torch.zeros(B, K, H, device=dev), torch.zeros(B, K, Lt, device=dev)
        used = torch.zeros(B, K, M, dtype=torch.bool, device=dev)
        kept = torch.zeros(B, K, dtype=torch.long, device=dev)
        tok = torch.full((B, K), -1, dtype=torch.long, device=dev)
        score, phi, kkey = (torch.full((B, K), -math.inf, device=dev) for _ in range(3))
        score[:, 0] = phi[:, 0] = 0
        kv = int(key.item()) & 0xFFFFFFFFFFFFFFFF                  # the root's key: a Gumbel(0) draw of the counter B S K M + b
        c0 = ((B * steps * K * M + np.arange(B, dtype=np.uint64)) & 0xFFFFFFFF).astype(np.uint32)
        u0 = ((_hash32(c0, kv & 0xFFFFFFFF, kv >> 32) >> np.uint32(9)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -23)
        kkey[:, 0] = -torch.log(-torch.log(torch.from_numpy(u0).to(dev)))
        stat = torch.full((B, K), EMPTY, dtype=torch.long, device=dev)
        stat[:, 0] = LIVE
        out = {n: [] for n in ("tokens", "parents", "scores", "probs", "phi", "keys")}
        slot = torch.arange(K, device=dev).view(1, K, 1).expand(B, K, M)
        sent_of = torch.arange(M, device=dev).view(1, 1, M).expand(B, K, M)
        for s in range(steps):
            p = torch.zeros(B, K, M, device=dev)
            hn, cn, vn = torch.zeros_like(h), torch.zeros_like(cell), torch.zeros_like(cov)
            for k in range(K):
                sent = emb.new_zeros(B, emb.shape[2]) if s == 0 else emb[rows, tok[:, k].clamp(0, Lt - 1)]
                o = ops.decoder_step_fwd(seq, sent.contiguous(), h[:, k].contiguous(), cell[:, k].contiguous(), cov[:, k].contiguous(),
                                         mask_u8)
                p[:, k], hn[:, k], cn[:, k], vn[:, k] = o[0], o[1], o[2], o[4]
            elig = _eligible(mask.bool().unsqueeze(1).expand(B, K, M), eos.view(B, 1).expand(B, K), used, kept, no_repeat,
                             min_sentences)
            cand = (stat == LIVE).unsqueeze(2) & (p > 0) & elig
            # the normaliser: mu, the integer masses, lam
            l = torch.log(p) * inv
            mu = torch.where(cand, l, ninf).max(2).values
            q = torch.where(cand, torch.floor(torch.exp(l - mu.unsqueeze(2)) * 16777216.0), torch.zeros_like(l)).long()
            lam = mu + torch.log(q.sum(2).float() * 5.9604644775390625e-08)
            phi2 = phi.unsqueeze(2) + (l - lam.unsqueeze(2))
            u = _uniforms(key, B, steps, s, K, M).to(dev)
            G = phi2 + -torch.log(-torch.log(u))
            Z = torch.where(cand, G, ninf).max(2).values
            a = G - Z.unsqueeze(2)
            l1 = torch.where(a > NEG_LN2, torch.log(-torch.expm1(a)), torch.log1p(-torch.exp(a)))
            v = (kkey.unsqueeze(2) - G) + l1
            ck = (kkey.unsqueeze(2) - torch.clamp_min(v, 0.0)) - torch.log1p(torch.exp(-v.abs()))
            c_key = torch.cat([torch.where(cand, ck, ninf).reshape(B, -1), kkey], 1)
            c_score = torch.cat([(score.unsqueeze(2) + torch.log(p)).reshape(B, -1), score], 1)
            c_phi = torch.cat([phi2.reshape(B, -1), phi], 1)
            c_p = torch.cat([p.reshape(B, -1), torch.ones(B, K, device=dev)], 1)
            c_par = torch.cat([slot.reshape(B, -1), torch.arange(K, device=dev).expand(B, K)], 1)
            c_tok = torch.cat([sent_of.reshape(B, -1), eos.view(B, 1).expand(B, K)], 1)
            c_ok = torch.cat([cand.reshape(B, -1), stat == DONE], 1)
            c_carry = torch.cat([torch.zeros(B, K * M, dtype=torch.bool, device=dev), stat == DONE], 1)
            order = torch.arange(c_key.shape[1], device=dev).expand(B, -1)
            for sk, desc in ((c_tok, False), (c_par, False), (c_p, True), (c_key, True), (c_ok.to(torch.int8), True)):
                _, idx = torch.sort(sk.gather(1, order), dim=1, descending=desc, stable=True)
                order = order.gather(1, idx)
            nxt = order[:, K:K + 1]                         # the threshold: the largest (K + 1)-th entry over the steps
            pruned = torch.where(c_ok.gather(1, nxt), c_key.gather(1, nxt), ninf).squeeze(1)
            kappa = pruned if s == 0 else torch.maximum(kappa, pruned)
            top = order[:, :K]
            ok = c_ok.gather(1, top)
            par = c_par.gather(1, top)
            t = c_tok.gather(1, top)
            carry = c_carry.gather(1, top)
            from_live = ok & ~carry
            out["tokens"].append(torch.where(ok, t, -1))
            out["parents"].append(torch.where(ok, par, -1).to(torch.int32))
            out["probs"].append(p.gather(1, par.view(B, K, 1).expand(B, K, M)) * from_live.unsqueeze(2))
            score, phi, kkey = (torch.where(ok, c.gather(1, top), ninf) for c in (c_score, c_phi, c_key))
            out["scores"].append(score)
            out["phi"].append(phi)
            out["keys"].append(kkey)
            g = par.view(B, K, 1)
            h, cell, cov = hn.gather(1, g.expand(B, K, H)), cn.gather(1, g.expand(B, K, H)), vn.gather(1, g.expand(B, K, Lt))
            below = t < eos.view(B, 1)
            used = used.gather(1, g.expand(B, K, M)) | ((sent_of == t.unsqueeze(2)) & below.unsqueeze(2))
            kept = kept.gather(1, par) + below.long()
            tok = torch.where(ok, t, -1)
            stat = torch.where(~ok, EMPTY, torch.where(carry | (t == eos.view(B, 1)), DONE, LIVE))
        res = {n: torch.stack(x, 1) for n, x in out.items()}
        res["kappa"] = kappa
        # every final slot walked back to step 0 (an empty slot: eos at every step)
        paths = torch.empty(B, K, steps, dtype=torch.long, device=dev)
        j = torch.arange(K, device=dev).expand(B, K).clone()
        empty = res["parents"][:, -1] < 0
        for s in range(steps - 1, -1, -1):
            paths[:, :, s] = torch.where(empty, eos.view(B, 1), res["tokens"][:, s].gather(1, j.clamp_min(0)))
            j = res["parents"][:, s].long().gather(1, j.clamp_min(0))
        res["paths"] = paths
        return res


def _run(model, b, steps, K, T, no_repeat, min_sentences, seed=11):
    from mmbidaf_b200 import ops
    emb, h0, enc_a, enc_i, mask, lens = _decoder_inputs(model, b)
    key = ops.seed_key(seed, "cuda")
    got = model.multimodal_att_decoder.beam_sample(emb, h0, enc_a, enc_i, mask, lens, steps, K, key, T, no_repeat, min_sentences)
    return (emb, h0, enc_a, enc_i, mask, lens, key), dict(zip(("tokens", "parents", "scores", "probs", "phi", "keys", "paths",
                                                               "path_slots", "kappa"), got))


def _check_samples(got, lens, no_repeat, min_sentences):
    """Distinct token rows among the non-empty final slots of every video, and the constraints in every sample."""
    paths, empty = got["paths"].cpu(), (got["path_slots"][:, :, -1] < 0).cpu()
    for v in range(paths.shape[0]):
        rows = [tuple(r) for r, e in zip(paths[v].tolist(), empty[v].tolist()) if not e]
        assert len(set(rows)) == len(rows) >= 1
        for r in rows:
            chosen = _select(r, int(lens[v]))
            if no_repeat:
                assert len(set(chosen)) == len(chosen)
            assert len(chosen) >= min(min_sentences, len(r), int(lens[v]) - 1)


@pytest.mark.parametrize("tier", ["fp32", "fast"], indirect=True)
@pytest.mark.parametrize("B", [1, 21])
@pytest.mark.parametrize("K", [1, 2, 4, 8])
@pytest.mark.parametrize("T", [1.0, 0.7])
@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
def test_beam_sample_equals_the_host_loop(tier, B, K, T, no_repeat, min_sentences):
    model = _model(64)
    b = _batch(B).to("cuda")
    inputs, got = _run(model, b, 16, K, T, no_repeat, min_sentences)
    want = _reference(model.multimodal_att_decoder, *inputs[:6], 16, K, inputs[6], T, no_repeat, min_sentences)
    for name in ("tokens", "parents", "scores", "phi", "keys", "probs", "paths", "kappa"):
        assert torch.equal(got[name], want[name]), name
    # the path slots walk the parents; the final slots are ranked by key
    B_, S = got["tokens"].shape[:2]
    j = torch.arange(K, device="cuda").expand(B_, K).clone()
    for s in range(S - 1, -1, -1):
        assert torch.equal(got["path_slots"][:, :, s].long(), torch.where(got["parents"][:, -1] < 0, -1, j))
        j = got["parents"][:, s].long().gather(1, j.clamp_min(0))
    keys = got["keys"][:, -1].nan_to_num(neginf=-3e38)
    assert (keys[:, :-1] >= keys[:, 1:]).all()
    _check_samples(got, b.text_len, no_repeat, min_sentences)
    if B > 1 and no_repeat:                                # the two-row transcript under min_sentences: [0, EOS, ..] alone
        assert int((got["path_slots"][1, :, -1] >= 0).sum()) == 1 and float(got["kappa"][1]) == -math.inf


def test_long_lecture_beam_sample_equals_the_host_loop(monkeypatch):
    from mmbidaf_b200 import ops
    model = _model(700)
    b = make_batch(32, 700, 60, 6, 6, seed=41).to("cuda")
    assert ops.decoder_cut(32, 700) == "chunks"            # the stochastic beam runs the cluster kernel; so must its reference
    monkeypatch.setenv("MMB_DECODER_CUT", "fused")
    for K, T, nr, ms in ((3, 1.0, True, 3), (2, 0.7, False, 0)):
        inputs, got = _run(model, b, 6, K, T, nr, ms)
        want = _reference(model.multimodal_att_decoder, *inputs[:6], 6, K, inputs[6], T, nr, ms)
        for name in ("tokens", "parents", "scores", "phi", "keys", "probs", "paths", "kappa"):
            assert torch.equal(got[name], want[name]), name
        _check_samples(got, b.text_len, nr, ms)


def _tiny(B):
    """B copies of a video of two sentences and the EOS row."""
    b = make_batch(1, 37, 45, 7, 3, seed=9)
    _short(b, 0, 3)
    return b


def _enumerate(eos, probs_of):
    """Every sequence of the no_repeat rule on a 2-sentence video over 3 steps, with its probability under the renormalised p (T = 1)
    from ``probs_of(prefix)`` -- the step distribution after that prefix -- in fp64."""
    seqs = {}

    def walk(prefix, pr):
        if len(prefix) == 3 or (prefix and prefix[-1] == eos):
            seqs[tuple(prefix)] = pr
            return
        p = probs_of(tuple(prefix))
        cand = [m for m in range(eos + 1) if (m == eos or m not in prefix) and p[m] > 0]
        tot = sum(p[m] for m in cand)
        for m in cand:
            walk(prefix + [m], pr * p[m] / tot)
    walk([], 1.0)
    return seqs


def test_complete_enumeration_of_a_tiny_video():
    from mmbidaf_b200 import ops
    model = _model(64)
    b = _tiny(1).to("cuda")
    inputs, got = _run(model, b, 3, 8, 1.0, True, 0)
    eos = 2
    nonempty = got["path_slots"][0, :, -1] >= 0
    assert int(nonempty.sum()) == 5 and not nonempty[5:].any()
    assert float(got["kappa"][0]) == -math.inf
    inc = Inclusion(got["phi"][:, -1], got["keys"][:, -1], got["kappa"])
    assert torch.equal(inc.probabilities()[0, :5], torch.ones(5, dtype=torch.float64, device="cuda"))
    w = inc.weights(normalise=False)[0]
    assert torch.equal(w[:5], torch.exp(got["phi"][0, -1, :5].double())) and (w[5:] == 0).all()
    assert abs(float(torch.exp(got["phi"][0, -1, :5].double()).sum()) - 1) < 1e-5
    # the probability of every sequence from the host loop's per-step p along its path
    ref = _reference(model.multimodal_att_decoder, *inputs[:6], 3, 8, inputs[6], 1.0, True, 0)
    rows = {}
    P, par, tok = ref["probs"][0].double().cpu(), ref["parents"][0].cpu(), ref["tokens"][0].cpu()
    for j in range(8):
        for s in range(3):
            if int(par[s, j]) < 0 or int(tok[s, j]) < 0 or not P[s, j].any():
                continue
            prefix, k = [], j                               # the prefix that produced row (s, j): walk back from step s - 1
            k = int(par[s, j])
            for s2 in range(s - 1, -1, -1):
                prefix.append(int(tok[s2, k]))
                k = int(par[s2, k])
            rows[tuple(reversed(prefix))] = P[s, j].tolist()
    seqs = _enumerate(eos, lambda prefix: rows[prefix])
    assert len(seqs) == 5
    got_seqs = {}
    for j in range(5):
        row = got["paths"][0, j].tolist()
        cut = row.index(eos) + 1 if eos in row else 3
        got_seqs[tuple(row[:cut])] = math.exp(float(got["phi"][0, -1, j]))
    assert set(got_seqs) == set(seqs)
    for sq, pr in seqs.items():
        assert abs(got_seqs[sq] - pr) <= 1e-5 * max(pr, 1e-3), (sq, got_seqs[sq], pr)


def test_pair_distribution_and_unbiased_estimate():
    """B = 4096 copies of the tiny video in one launch (independent counters), K = 2: the ordered pair (slot 0, slot 1) follows
    pi_i pi_j / (1 - pi_i), and the importance-weighted estimate of an indicator matches its expectation."""
    from scipy import stats
    from mmbidaf_b200 import ops
    model = _model(64)
    b = _tiny(1).to("cuda")
    inputs1, full = _run(model, b, 3, 8, 1.0, True, 0)
    eos = 2
    pi = {}
    for j in range(5):
        row = full["paths"][0, j].tolist()
        pi[tuple(row[:row.index(eos) + 1] if eos in row else row)] = math.exp(float(full["phi"][0, -1, j].double()))
    n = 4096
    emb, h0, enc_a, enc_i, mask, lens = (t.expand(n, *t.shape[1:]).contiguous() for t in inputs1[:6])
    key = ops.seed_key(2024, "cuda")
    got = model.multimodal_att_decoder.beam_sample(emb, h0, enc_a, enc_i, mask, lens, 3, 2, key, 1.0, True, 0)
    paths, phi, keys, kappa = got[6].cpu().tolist(), got[4][:, -1], got[5][:, -1], got[8]

    def seq(row):
        return tuple(row[:row.index(eos) + 1] if eos in row else row)
    names = sorted(pi)
    counts = np.zeros((5, 5))
    for r in paths:
        counts[names.index(seq(r[0])), names.index(seq(r[1]))] += 1
    expect = np.array([[pi[a] * pi[c] / (1 - pi[a]) if a != c else 0.0 for c in names] for a in names]) * n
    assert counts[np.eye(5, dtype=bool)].sum() == 0                # distinct
    off = ~np.eye(5, dtype=bool)
    e, o = expect[off], counts[off]
    big = e >= 5                                                 # pool the rare pairs into one bin
    e2, o2 = np.append(e[big], e[~big].sum()), np.append(o[big], o[~big].sum())
    if e2[-1] == 0:
        e2, o2 = e2[:-1], o2[:-1]
    assert stats.chisquare(o2, e2 * o2.sum() / e2.sum()).pvalue > 1e-3
    # f(y) = 1 when sentence 0 is in the summary: E[f] = the mass of those sequences; sum_i w_i f(y_i) per copy, unnormalised weights
    f = lambda sq: 1.0 if 0 in sq else 0.0
    exact = sum(p for sq, p in pi.items() if f(sq))
    w = Inclusion(phi, keys, kappa).weights(normalise=False).cpu().numpy()
    fy = np.array([[f(seq(r[0])), f(seq(r[1]))] for r in paths])
    est = (w * fy).sum(1)
    assert abs(est.mean() - exact) <= 4 * est.std() / math.sqrt(n), (est.mean(), exact, est.std())


@pytest.mark.parametrize("no_repeat,min_sentences", [(False, 0), (True, 3)])
@pytest.mark.parametrize("T", [1.0, 0.7])
def test_width_one_is_num_samples_one(no_repeat, min_sentences, T):
    """Same key, same counters: the picks equal those of num_samples=1 up to each video's first EOS.  Where a pick differs, the two
    best candidates' perturbed scores of that step are within fp32 rounding of each other."""
    model = _model(64)
    b = _batch(21).to("cuda")
    inputs, got = _run(model, b, 16, 1, T, no_repeat, min_sentences)
    emb, h0, enc_a, enc_i, mask, lens, key = inputs
    probs, tokens = model.multimodal_att_decoder.sample(emb, h0, enc_a, enc_i, mask, lens, 16, 1, key, T, 0, no_repeat, min_sentences)
    bs, sm = got["paths"][:, 0].cpu(), tokens[:, 0].cpu()
    inv = float(np.float32(1.0) / np.float32(T))
    differ = 0
    for v in range(bs.shape[0]):
        eos = int(lens[v]) - 1
        for s in range(16):
            if int(bs[v, s]) != int(sm[v, s]):
                # the same prefix gave the same distribution: the scores of the candidates of that step
                p = probs[v, 0, s]
                u = _uniforms(key, bs.shape[0], 16, s, 1, p.shape[0])[v, 0].cuda()
                z = torch.log(p) * inv - torch.log(-torch.log(u))
                a, c = float(z[int(bs[v, s])]), float(z[int(sm[v, s])])
                # (the stochastic beam adds the path's phi before it compares: rounding at that magnitude)
                mag = max(abs(a), abs(c), abs(float(got["phi"][v, s - 1, 0])) if s else 0.0, 1.0)
                assert abs(a - c) <= 8 * np.spacing(np.float32(mag)), (v, s, a, c)
                differ += 1
                break
            if int(bs[v, s]) == eos:
                break
    assert differ <= 2


def test_summarize_and_summarizer_replays():
    from mmbidaf_b200.summarize import Summarizer
    model = _model(64)
    b = _batch(4).to("cuda")
    kw = dict(num_samples=4, replacement=False, temperature=0.7, seed=3)
    s1 = model.summarize(b.text, b.text_len, b.audio, b.audio_len, b.images, b.image_len, 12, **kw)
    assert s1.samples.tokens.shape == (4, 4, 12) and s1.inclusion is not None and s1.beams is None
    # the summary is the likeliest sample's, and every sample's summary follows its path
    lists = s1.samples.summaries(b.text_len)
    best = s1.samples.logp.argmax(1).tolist()
    assert s1.to_lists() == [lists[v][best[v]][0] for v in range(4)]
    summarizer = Summarizer(model)
    batches = [make_batch(4, 37, 45, 7, 12, seed=s).to("cuda") for s in (1, 2)]
    for bb in batches:
        got = summarizer(bb, **kw)
        got = [t.clone() for t in (got.indices, got.counts, got.samples.tokens, got.samples.probs, got.samples.logp,
                                   *got.inclusion)]
        w = model.summarize(bb.text, bb.text_len, bb.audio, bb.audio_len, bb.images, bb.image_len, bb.max_dec_len, **kw)
        want = (w.indices, w.counts, w.samples.tokens, w.samples.probs, w.samples.logp, *w.inclusion)
        assert all(torch.equal(g, x) for g, x in zip(got, want))
    assert len(summarizer.buckets) == 1
    summarizer(batches[0], num_samples=4, temperature=0.7, seed=3)             # with replacement: its own bucket
    assert len(summarizer.buckets) == 2
    fresh = dict(num_samples=4, replacement=False)                              # seed None: a fresh key on every replay
    r1 = summarizer(batches[0], **fresh).samples.tokens.clone()
    r2 = summarizer(batches[0], **fresh).samples.tokens.clone()
    assert len(summarizer.buckets) == 3 and not torch.equal(r1, r2)
