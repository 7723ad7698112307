"""Attention blocks of the MMBiDAF hot path on B200.

Same public surface as the reference's layers/attention.py: ``BiDAFAttention``, ``masked_softmax``,
``MultimodalAttentionDecoder`` with identical constructor / ``forward`` signatures, parameter names and
shapes.  The arithmetic runs in the fused sm_100a kernels of csrc/ (bidaf_*.cu, decoder_fwd.cu,
masked_softmax.cu); nothing here falls back to a CPU or library implementation of those ops.
"""
from __future__ import annotations

import weakref

import torch
import torch.nn as nn
import torch.nn.functional as F  # noqa: F401

from .. import functional as Fn
from .. import ops

__all__ = ["BiDAFAttention", "masked_softmax", "MultimodalAttentionDecoder"]


def _lib_fields():
    from .._lib import DECODER_WEIGHT_FIELDS
    return DECODER_WEIGHT_FIELDS


def _lin(attr, part):
    return lambda m: getattr(getattr(m, attr), part)


# C-ABI field (struct mmb_decoder_weights) -> module parameter
_FIELD_TO_PARAM = {}
for _f, _attr in (("W2", "W2"), ("Wc1", "Wc1"), ("v1", "v1"), ("W4", "W4"), ("Wc2", "Wc2"), ("v2", "v2")):
    _FIELD_TO_PARAM[_f] = _lin(_attr, "weight")
    _FIELD_TO_PARAM[("b" + _f[1:]) if _f[0] == "W" else _f + "b"] = _lin(_attr, "bias")
for _k in "1234":
    _FIELD_TO_PARAM["Wb" + _k] = _lin("W_beta_" + _k, "weight")
    _FIELD_TO_PARAM["bb" + _k] = _lin("W_beta_" + _k, "bias")
for _k in "12":
    _FIELD_TO_PARAM["vb" + _k] = _lin("v_beta_" + _k, "weight")
    _FIELD_TO_PARAM["vb" + _k + "b"] = _lin("v_beta_" + _k, "bias")
_FIELD_TO_PARAM.update({"lstm_w_ih": _lin("lstm", "weight_ih_l0"), "lstm_w_hh": _lin("lstm", "weight_hh_l0"),
                        "lstm_b_ih": _lin("lstm", "bias_ih_l0"), "lstm_b_hh": _lin("lstm", "bias_hh_l0"),
                        "out_w": _lin("out", "weight"), "out_b": _lin("out", "bias")})


def _keep_masks(shapes, drop_prob, device):
    """Bernoulli(1-p) keep masks as uint8, one per shape: the library's counter-based bits (one key launch + one mask launch each;
    csrc/common.cuh::dropout_keep), not ATen's Philox stream -- parity GIVEN the masks is what the tests check."""
    keys = ops.rng_next_keys(device, len(shapes))
    return tuple(ops.dropout_mask_u8(keys[i:i + 1], 1.0 - drop_prob, tuple(shape)) for i, shape in enumerate(shapes))


class BiDAFAttention(nn.Module):
    """Bidirectional text<->modality attention (reference attention.py:9-75).

    forward(text (B,Lc,d), modality (B,Lq,d), text_mask (B,Lc), modality_mask (B,Lq)) -> (B,Lc,4d)
    = [text, a, text*a, text*b].  ``precision`` selects the contraction tier of the fused kernel
    ("fp32": rel <= 1e-5; "bf16": tcgen05 tensor cores, rel <= 2e-2)."""

    precision = "fp32"

    def __init__(self, hidden_size, drop_prob=0.1):
        super().__init__()
        self.drop_prob = drop_prob
        self.text_weight = nn.Parameter(torch.zeros(hidden_size, 1))
        self.modality_weight = nn.Parameter(torch.zeros(hidden_size, 1))
        self.text_modality_weight = nn.Parameter(torch.zeros(1, 1, hidden_size))
        for weight in (self.text_weight, self.modality_weight, self.text_modality_weight):
            nn.init.xavier_uniform_(weight)
        self.bias = nn.Parameter(torch.zeros(1))

    def predraw_dropout(self, text_shape, modality_shape, device):
        """Optional: draw this call's keep-masks NOW (on the current stream) -- they depend on shapes only, so a caller that knows
        the shapes ahead (mmbidaf_b200/models.py: while the encoders still run) takes two mask draws off the serial chain between
        the encoders and the fused kernel.  Consumed by the next ``forward`` with matching shapes; same draw order (text, modality)."""
        self._predrawn = None
        if self.training and self.drop_prob > 0:
            self._predrawn = _keep_masks((text_shape, modality_shape), self.drop_prob, device)

    def _dropout_masks(self, text, modality):
        pre, self._predrawn = getattr(self, "_predrawn", None), None
        if not self.training or self.drop_prob <= 0:
            return None, None, 1.0
        if pre is not None and pre[0].shape == text.shape and pre[1].shape == modality.shape:
            return pre[0], pre[1], 1.0 / (1.0 - self.drop_prob)
        # same draw order as the reference: text first, then modality (attention.py:66-67)
        keep_c, keep_q = _keep_masks((text.shape, modality.shape), self.drop_prob, text.device)
        return keep_c, keep_q, 1.0 / (1.0 - self.drop_prob)

    def forward(self, text, modality, text_mask, modality_mask):
        if not text.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.BiDAFAttention runs on a B200 only (no CPU fallback)")
        keep_c, keep_q, scale = self._dropout_masks(text, modality)
        prec = ops.PREC_BF16 if self.precision == "bf16" else ops.PREC_FP32
        return Fn.bidaf_attention(text, modality, text_mask, modality_mask, self.text_weight, self.modality_weight,
                                  self.text_modality_weight, self.bias, keep_c, keep_q, scale, prec)

    def get_similarity_matrix(self, text, modality):
        """Materialised S (B,Lc,Lq).  Kept for API compatibility (attention.py:56-75); ``forward`` never
        calls it -- the fused kernel builds S tile by tile on chip."""
        text = F.dropout(text, self.drop_prob, self.training)
        modality = F.dropout(modality, self.drop_prob, self.training)
        s = torch.baddbmm(text @ self.text_weight + (modality @ self.modality_weight).transpose(1, 2),
                          text * self.text_modality_weight, modality.transpose(1, 2))
        return s + self.bias


def masked_softmax(logits, mask, dim=-1, log_softmax=False):
    """softmax(mask*x + (1-mask)*-1e30) along ``dim`` (reference attention.py:78-98), as a CUDA kernel."""
    return Fn.masked_softmax(logits, mask, dim, log_softmax)


class MultimodalAttentionDecoder(nn.Module):
    """Pointer-style decoder step with two coverage attentions (reference attention.py:100-186).

    forward(sent_embed (B,1,E), decoder_hidden (B,1,H), decoder_cell_state (1,B,H), text_audio_enc_out
    (B,Lt,2H), text_img_enc_out (B,Lt,2H), coverage_vec (B,Lt,1), mask (B,M)) -> (final_out (B,M),
    decoder_hidden (B,1,H), decoder_cell_state (1,B,H), att_cov_dist (B,Lt,1), coverage_vec (B,Lt,1)).

    ``W1(text_audio_enc_out)`` and ``W3(text_img_enc_out)`` do not change between steps; they are computed
    once per pair of encoder tensors and cached on the tensors' identity."""

    def __init__(self, text_embedding_size, hidden_size, output_size, num_layers=1, dropout=0.1):
        super().__init__()
        self.text_embedding_size = text_embedding_size
        self.hidden_size = hidden_size
        self.output_size = output_size
        self.num_layers = num_layers
        self.dropout = dropout
        h2 = 2 * hidden_size
        self.W1 = nn.Linear(h2, h2)
        self.W2 = nn.Linear(hidden_size, h2)
        self.Wc1 = nn.Linear(1, h2)
        self.v1 = nn.Linear(h2, 1)
        self.tanh = nn.Tanh()
        self.W3 = nn.Linear(h2, h2)
        self.W4 = nn.Linear(hidden_size, h2)
        self.Wc2 = nn.Linear(1, h2)
        self.v2 = nn.Linear(h2, 1)
        self.W_beta_1 = nn.Linear(h2, h2)
        self.W_beta_2 = nn.Linear(hidden_size, h2)
        self.W_beta_3 = nn.Linear(h2, h2)
        self.W_beta_4 = nn.Linear(hidden_size, h2)
        self.v_beta_1 = nn.Linear(h2, 1)
        self.v_beta_2 = nn.Linear(h2, 1)
        self.lstm = nn.LSTM(text_embedding_size + h2, hidden_size, num_layers, batch_first=True)
        self.out = nn.Linear(hidden_size, output_size)
        self.softmax = nn.Softmax()
        self._cache = None
        self._prepared = None

    def prepare(self):
        """Optional: lay this step's weights out for the decoder kernels NOW (on the current stream), e.g. while the
        encoders still run; the next new sequence picks the result up (once) instead of building it in front of its
        first step.  Must be called again after the weights change."""
        if self.W1.weight.is_cuda:
            params = {name: self._param_of(name) for name in _lib_fields()}
            self._prepared = ops.DecoderWeights(params, self.output_size)

    def hoist(self, which, enc):
        """Optional: compute the step-invariant projection of one encoder output NOW, on the current stream -- ``which`` = "a"
        (``W1 enc_a``, attention.py:152) or "i" (``W3 enc_i``, attention.py:157).  A caller that runs the two modality chains on
        their own streams (mmbidaf_b200/models.py) calls it at the end of each chain: the GEMM of the chain that finishes first is
        off the serial path in front of the first decoder step, and the two gradient GEMMs behind the last step run side by side
        (autograd replays a backward op on the stream of its forward).  The next new sequence over the same tensor picks the
        result up (once)."""
        lin = self.W1 if which == "a" else self.W3
        proj = Fn.tall_linear_bias(enc, lin.weight, lin.bias)
        if getattr(self, "_hoisted", None) is None:
            self._hoisted = {}
        self._hoisted[which] = (weakref.ref(enc), enc._version, torch.is_grad_enabled(), proj)
        return proj

    def _hoisted_or_new(self, which, enc, lin):
        hit = (getattr(self, "_hoisted", None) or {}).pop(which, None)
        if hit is not None and hit[0]() is enc and hit[1] == enc._version and hit[2] == torch.is_grad_enabled():
            return hit[3]
        return Fn.tall_linear_bias(enc, lin.weight, lin.bias)

    # ---- per-sequence state: step-invariant projections (+ the autograd tape when training) ----------------
    def _sequence(self, enc_a, enc_i):
        grad = torch.is_grad_enabled()
        c = self._cache
        if c is not None and c["a"]() is enc_a and c["i"]() is enc_i and c["key"] == (enc_a._version, enc_i._version, grad):
            return c
        # hoisted: the reference recomputes them per step (attention.py:152, 157)
        proj_a = self._hoisted_or_new("a", enc_a, self.W1)
        proj_i = self._hoisted_or_new("i", enc_i, self.W3)
        c = {"a": weakref.ref(enc_a), "i": weakref.ref(enc_i), "key": (enc_a._version, enc_i._version, grad),
             "proj_a": proj_a, "proj_i": proj_i, "seq": None, "tape": None, "token": None, "last_h": None}
        params = {name: self._param_of(name) for name in _lib_fields()}
        prepared, self._prepared = self._prepared, None             # used at most once: the weights move every training step
        c["seq"] = ops.DecoderSeq(params, enc_a, enc_i, proj_a, proj_i, self.output_size, weights=prepared)
        needs_grad = grad and (proj_a.requires_grad or enc_a.requires_grad or enc_i.requires_grad)
        if needs_grad:
            tape = Fn.DecoderTape(c["seq"])
            c["tape"], c["token"] = tape, Fn.decoder_open(tape, proj_a, proj_i, enc_a, enc_i, list(params.values()))
        self._cache = c
        return c

    def _param_of(self, field):
        return _FIELD_TO_PARAM[field](self)

    def forward(self, sent_embed, decoder_hidden, decoder_cell_state, text_audio_enc_out, text_img_enc_out,
                coverage_vec, mask):
        return self.step(sent_embed, decoder_hidden, decoder_cell_state, text_audio_enc_out, text_img_enc_out,
                         coverage_vec, mask)[:5]

    def greedy(self, emb_text, h0, enc_a, enc_i, mask, steps, target=None, text_len=None, no_repeat=False, min_sentences=0):
        """The greedy decode of ``steps`` steps in eval mode (models.py:145-199, the ``else`` branches), batched: start from h0
        (B, H) or (B, 1, H), a zero cell, coverage and input row; each step's arg-max row of ``emb_text`` (B, Lt, E) is the next
        input.  ``target`` (B, T) with T >= steps is optional.  No autograd.  Returns (out_distributions (B, steps, M), argmax
        (B, steps) int64, loss_terms (steps, 2, B) = per step [nll | coverage term] or None) -- bit for bit what ``steps`` calls of
        :meth:`step` with an arg-max and a gather in between give.  Where the decoder step runs as one cluster kernel
        (``ops.decoder_cut``) the whole roll-out is one launch; long lectures run the chunk-parallel cut step by step.
        ``no_repeat`` / ``min_sentences`` constrain the pick (the rule at mmb_decoder_greedy_constrained_fused in
        include/mmbidaf_b200.h; ``text_len`` (B) gives each video's EOS row, text_len - 1): the roll-out is then always one launch of
        the cluster kernel, takes no ``target`` and returns None as loss_terms."""
        if not enc_a.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        constrained = bool(no_repeat) or min_sentences != 0
        if constrained and (target is not None or text_len is None):
            raise ValueError("greedy: a constrained roll-out needs text_len and takes no target (the eval loss is the unconstrained "
                             "roll-out's)")
        with torch.no_grad():
            seq = self._sequence(enc_a, enc_i)["seq"]
            B, Lt = seq.B, seq.Lt
            emb = emb_text.contiguous()
            h = h0.reshape(B, -1).contiguous()
            mask_u8 = ops._u8(mask)
            if constrained:
                probs, picks = ops.decoder_greedy_constrained_fwd(seq, emb, h, mask_u8, text_len.to(torch.int32).contiguous(), steps,
                                                                  no_repeat, min_sentences)
                return probs, picks, None
            tgt = None if target is None else target.reshape(B, -1).to(torch.int64).contiguous()
            if ops.decoder_cut(B, Lt) != "chunks":
                return ops.decoder_greedy_fwd(seq, emb, h, mask_u8, steps, tgt)
            if tgt is not None and tgt.shape[1] < steps:
                raise ValueError(f"greedy: {tgt.shape[1]} targets for {steps} steps")
            rows = torch.arange(B, device=h.device)
            sent = emb.new_zeros(B, emb.shape[2])
            cell = h.new_zeros(B, seq.H)
            cov = h.new_zeros(B, Lt)
            probs, picks, terms = [], [], []
            for s in range(steps):
                p, h, cell, _, cov, am, _, lossvec = ops.decoder_step_fwd(
                    seq, sent, h, cell, cov, mask_u8, want_argmax=True, target=None if tgt is None else tgt[:, s].contiguous())
                sent = emb[rows, am]                                           # models.py:184,:193
                probs.append(p)
                picks.append(am)
                terms.append(lossvec)
            return torch.stack(probs, 1), torch.stack(picks, 1), (torch.stack(terms) if tgt is not None else None)

    def force(self, emb_text, h0, enc_a, enc_i, mask, tokens, want_probs=False):
        """The teacher-forced decode of given token rows in eval mode: ``tokens`` (B, N, S) int64, N (1..64) candidates per video,
        each run as :meth:`greedy` runs with its own tokens as the picks (the rule at mmb_decoder_forced_fused in
        include/mmbidaf_b200.h), as ONE launch of the cluster kernel whatever ``ops.decoder_cut`` says.  Same start as :meth:`greedy`.
        No autograd.  Returns ``ops.decoder_forced_fwd``'s (probs (B,N,S,M) or None, p_tok (B,N,S), loss_terms (S,2,B N))."""
        if not enc_a.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        with torch.no_grad():
            seq = self._sequence(enc_a, enc_i)["seq"]
            B = seq.B
            return ops.decoder_forced_fwd(seq, emb_text.contiguous(), h0.reshape(B, -1).contiguous(), ops._u8(mask),
                                          tokens.contiguous(), want_probs)

    def force_train(self, emb_text, h0, enc_a, enc_i, mask, tokens):
        """:meth:`force` under autograd: (p_tok (B,N,S), loss_terms (S,2,B N)) with gradients into ``enc_a`` / ``enc_i`` (also through
        the hoisted W1 / W3 projections), ``h0`` and every decoder parameter -- one launch forward, one launch backward (the rules at
        mmb_decoder_forced_train_fused / mmb_decoder_forced_bwd_fused in include/mmbidaf_b200.h), whatever ``ops.decoder_cut`` says.
        No gradient reaches ``emb_text``.  The sequence is its own: the per-step tape of :meth:`step` is not used."""
        if not enc_a.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        proj_a = self._hoisted_or_new("a", enc_a, self.W1)
        proj_i = self._hoisted_or_new("i", enc_i, self.W3)
        params = {name: self._param_of(name) for name in _lib_fields()}
        prepared, self._prepared = self._prepared, None
        seq = ops.DecoderSeq(params, enc_a, enc_i, proj_a, proj_i, self.output_size, weights=prepared)
        return Fn.decoder_forced(seq, emb_text.detach().contiguous(), ops._u8(mask), tokens.contiguous(), proj_a, proj_i, enc_a, enc_i,
                                 h0.reshape(seq.B, -1), list(params.values()))

    def beam(self, emb_text, h0, enc_a, enc_i, mask, text_len, steps, width, no_repeat=False, min_sentences=0):
        """The beam decode of ``steps`` steps in eval mode with ``width`` (1..8) hypotheses per video, as ONE launch of the cluster
        kernel whatever ``ops.decoder_cut`` says (there is no chunk-cut beam); the rule is documented at mmb_decoder_beam_fused in
        include/mmbidaf_b200.h, and with ``no_repeat`` / ``min_sentences`` at mmb_decoder_beam_constrained_fused.  Same start as
        :meth:`greedy`; ``text_len`` (B) int32 gives each video's EOS row (text_len - 1).
        No autograd.  Returns ``ops.decoder_beam_fwd``'s (tokens, parents, scores, probs, best, path)."""
        if not enc_a.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        with torch.no_grad():
            seq = self._sequence(enc_a, enc_i)["seq"]
            B = seq.B
            return ops.decoder_beam_fwd(seq, emb_text.contiguous(), h0.reshape(B, -1).contiguous(), ops._u8(mask),
                                        text_len.to(torch.int32).contiguous(), steps, width, no_repeat, min_sentences)

    def beam_sample(self, emb_text, h0, enc_a, enc_i, mask, text_len, steps, width, key, temperature=1.0, no_repeat=False,
                    min_sentences=0):
        """The stochastic beam decode of ``steps`` steps in eval mode: ``width`` (1..8) distinct sequences per video, a sample without
        replacement from p^(1/``temperature``) renormalised over the candidates (the constraints included), as ONE launch of the
        cluster kernel whatever ``ops.decoder_cut`` says; the rule (the keys, the counter of ``key``, the threshold) is documented at
        mmb_decoder_beam_sample_fused in include/mmbidaf_b200.h.  Same start as :meth:`greedy`; ``text_len`` (B) int32 gives each
        video's EOS row; ``key`` (1) int64 on the device.  No autograd.  Returns ``ops.decoder_beam_sample_fwd``'s (tokens, parents,
        scores, probs, phi, keys, paths, path_slots, kappa)."""
        if not enc_a.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        with torch.no_grad():
            seq = self._sequence(enc_a, enc_i)["seq"]
            B = seq.B
            return ops.decoder_beam_sample_fwd(seq, emb_text.contiguous(), h0.reshape(B, -1).contiguous(), ops._u8(mask),
                                               text_len.to(torch.int32).contiguous(), steps, width, key, temperature, no_repeat,
                                               min_sentences)

    def sample(self, emb_text, h0, enc_a, enc_i, mask, text_len, steps, num_samples, key, temperature=1.0, top_k=0, no_repeat=False,
               min_sentences=0, *, top_p=1.0):
        """``num_samples`` sampled decodes of ``steps`` steps per video in eval mode, as ONE launch of the cluster kernel whatever
        ``ops.decoder_cut`` says; the rule (temperature, top_k, the constraints, the counter of ``key``) is documented at
        mmb_decoder_sample_fused in include/mmbidaf_b200.h, and ``top_p`` < 1 (the nucleus) at mmb_decoder_sample_nucleus_fused.  Same
        start as :meth:`greedy`; ``text_len`` (B) int32 gives each video's EOS row; ``key`` (1) int64 on the device.  No autograd.
        Returns ``ops.decoder_sample_fwd``'s (probs (B,N,S,M), tokens (B,N,S))."""
        if not enc_a.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        with torch.no_grad():
            seq = self._sequence(enc_a, enc_i)["seq"]
            B = seq.B
            return ops.decoder_sample_fwd(seq, emb_text.contiguous(), h0.reshape(B, -1).contiguous(), ops._u8(mask),
                                          text_len.to(torch.int32).contiguous(), steps, num_samples, key, temperature, top_k,
                                          no_repeat, min_sentences, top_p)

    def step(self, sent_embed, decoder_hidden, decoder_cell_state, text_audio_enc_out, text_img_enc_out, coverage_vec,
             mask, target=None):
        """``forward`` plus, when ``target`` (B) int64 is given, the step's fused loss terms as a sixth result:
        (2, B) = [-log(final_out[b, target[b]] + 1e-12), sum_t min(att_cov_dist, coverage_vec)] (models.py:168-178)."""
        if not text_audio_enc_out.is_cuda:
            raise RuntimeError("mmbidaf_b200.layers.MultimodalAttentionDecoder runs on a B200 only (no CPU fallback)")
        if self.num_layers != 1:
            raise RuntimeError("MultimodalAttentionDecoder: only num_layers=1 is supported (the reference model uses 1)")
        seq = self._sequence(text_audio_enc_out, text_img_enc_out)
        B, Lt, _ = text_audio_enc_out.shape
        sent = sent_embed.reshape(B, -1).contiguous()
        h = decoder_hidden.reshape(B, -1).contiguous()
        cell = decoder_cell_state.reshape(B, -1).contiguous()
        cov = coverage_vec.reshape(B, Lt).contiguous()
        tgt = None if target is None else target.reshape(B).to(torch.int64).contiguous()
        if seq["tape"] is not None:
            # The token makes the sequence's closing backward (_DecoderOpen) run after this step's.  When the step continues
            # the previous one (its hidden state is that step's output, as in models.py:163) the chain of hidden-state
            # gradients already orders it behind a step that holds the token, so only the first step of a chain takes it:
            # no per-step gradient accumulation on the token.
            # (decided by tensor identity -- the step's hidden state is the previous step's output or a view of it -- not by address:
            # the caching allocator can hand an unrelated tensor the address of a freed one)
            prev = seq["last_h"]
            chained = prev is not None and (h is prev or h._base is prev)
            probs, h, cell, att, cov, lossvec = Fn.decoder_step(seq["tape"], None if chained else seq["token"], sent, h, cell,
                                                                cov, ops._u8(mask), tgt)
            seq["last_h"] = h
        else:
            probs, h, cell, att, cov, _, _, lossvec = ops.decoder_step_fwd(seq["seq"], sent, h, cell, cov, ops._u8(mask),
                                                                           target=tgt)
        return probs, h.unsqueeze(1), cell.unsqueeze(0), att.unsqueeze(2), cov.unsqueeze(2), (lossvec if tgt is not None else None)
