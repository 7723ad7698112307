"""MMBiDAF on B200: the reference's ``models.MMBiDAF`` module surface over the fused kernels.

Constructor and ``forward`` signatures, sub-module names and every parameter name / shape equal the
reference's (models.py:29-83, :94), so ``train.py`` / ``evaluate.py`` style drivers and reference
checkpoints (with or without the DataParallel ``module.`` prefix) work unchanged.  Differences are all
inside ``forward``: masks are built on the device, and the decode loop gathers target probabilities and
next inputs with device-side indexing instead of ``B x T`` ``int(tensor)`` host round trips
(reference models.py:166-173, :186-193).  The value of every returned quantity is the reference's.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from . import functional as Fn
from . import ops
from .layers import BiDAFAttention, Embedding, ImageEmbedding, MultimodalAttentionDecoder, RNNEncoder

__all__ = ["MMBiDAF"]


class MMBiDAF(nn.Module):
    """Embedding -> bi-LSTM encoders -> BiDAF (text<->audio, text<->image) -> modality-aware 2-layer
    bi-LSTMs -> multimodal attention decoder with coverage -> distribution over source sentences."""

    def __init__(self, hidden_size, text_embedding_size, audio_embedding_size, image_embedding_size, device,
                 drop_prob=0., max_transcript_length=405):
        super().__init__()
        self.device = device
        self.max_transcript_length = max_transcript_length
        self.emb = Embedding(embedding_size=text_embedding_size, hidden_size=hidden_size, drop_prob=drop_prob)
        self.a_emb = Embedding(embedding_size=audio_embedding_size, hidden_size=hidden_size, drop_prob=drop_prob)
        self.i_emb = Embedding(embedding_size=image_embedding_size, hidden_size=hidden_size, drop_prob=drop_prob)
        self.text_enc = RNNEncoder(input_size=hidden_size, hidden_size=hidden_size, num_layers=1, drop_prob=drop_prob)
        self.audio_enc = RNNEncoder(input_size=hidden_size, hidden_size=hidden_size, num_layers=1, drop_prob=drop_prob)
        self.image_enc = RNNEncoder(input_size=hidden_size, hidden_size=hidden_size, num_layers=1, drop_prob=drop_prob)
        self.image_keyframes_emb = ImageEmbedding()
        self.bidaf_att_audio = BiDAFAttention(2 * hidden_size, drop_prob=drop_prob)
        self.bidaf_att_image = BiDAFAttention(2 * hidden_size, drop_prob=drop_prob)
        self.mod_t_a = RNNEncoder(input_size=8 * hidden_size, hidden_size=hidden_size, num_layers=2, drop_prob=drop_prob)
        self.mod_t_i = RNNEncoder(input_size=8 * hidden_size, hidden_size=hidden_size, num_layers=2, drop_prob=drop_prob)
        self.multimodal_att_decoder = MultimodalAttentionDecoder(text_embedding_size, hidden_size,
                                                                 max_transcript_length, num_layers=1)

    # Independent branches (three encoders; two BiDAF + modality-encoder chains) run on side streams so
    # that their latency-bound recurrences overlap on the 148 SMs.  autograd replays each backward op on
    # the stream of its forward op, so the overlap carries over to the backward pass.
    use_streams = True
    # the text / image encoders start behind the audio embedding (the audio chain is the critical path); MMB_NO_STAGGER=1: A/B measurements
    stagger_encoders = os.environ.get("MMB_NO_STAGGER", "0") != "1"

    def _fork_join(self, jobs, meanwhile=None):
        """Run ``jobs`` on side streams and join them into the current stream.  ``meanwhile`` (optional) is issued on the
        current stream between the fork and the join: glue that does not depend on the jobs' results (masks, decoder
        start state, per-step weight layouts) runs beside the recurrences instead of after them."""
        if not (self.use_streams and torch.cuda.is_available()):
            results = [job() for job in jobs]
            if meanwhile is not None:
                meanwhile()
            return results
        main = torch.cuda.current_stream()
        if getattr(self, "_streams", None) is None or self._streams[0].device != main.device:
            # the first job of a fork is the one on the critical path (the 1024-frame audio recurrence): its stream gets
            # the high priority, so its 64 CTAs are not queued behind the shorter text / image recurrences (192 CTAs
            # for 148 SMs) -- that ordering was a coin flip and made the step time bimodal
            object.__setattr__(self, "_streams", [torch.cuda.Stream(device=main.device, priority=-1 if i == 0 else 0)
                                                  for i in range(3)])
        results = []
        for stream, job in zip(self._streams, jobs):
            stream.wait_stream(main)
            with torch.cuda.stream(stream):
                results.append(job())
        if meanwhile is not None:
            meanwhile()
        capturing = torch.cuda.is_current_stream_capturing()
        for stream, res in zip(self._streams, results):
            main.wait_stream(stream)
            if capturing:
                continue                      # graph-private pool: lifetimes are fixed by the captured order
            for t in res:
                if isinstance(t, torch.Tensor):
                    t.record_stream(main)
        return results

    def load_state_dict(self, state_dict, strict=True, **kw):
        """Accepts reference checkpoints saved from ``nn.DataParallel`` (keys prefixed ``module.``)."""
        if state_dict and all(k.startswith("module.") for k in state_dict):
            state_dict = {k[len("module."):]: v for k, v in state_dict.items()}
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def get_mask(self, X, X_len):
        """bool (B, L): position < length, on X's device (reference models.py:86-92 builds it on the CPU)."""
        from .layers.encoding import length_plan
        return length_plan(X_len, X.device).mask(X.size(1))[0]      # one kernel from the device lengths (csrc/length_plan.cu)

    def forward(self, embedded_text, original_text_lengths, embedded_audio, original_audio_lengths, transformed_images,
                original_image_lengths, batch_target_indices, original_target_len, max_dec_len):
        B, Lt = embedded_text.size(0), embedded_text.size(1)
        steps = batch_target_indices.size(1) if self.training else max_dec_len
        start = {}

        def decoder_start():                     # everything the decode loop needs that does not depend on the encoders' output
            start["cell"] = embedded_text.new_zeros(1, B, self.mod_t_a.rnn.hidden_size)
            start["input"] = embedded_text.new_zeros(B, 1, embedded_text.size(-1))
            start["cov"] = embedded_text.new_zeros(B, Lt, 1)
            start["rows"] = torch.arange(B, device=embedded_text.device)
            start["targets"] = batch_target_indices.reshape(B, -1).to(embedded_text.device).long()   # int(tensor), models.py:168
            # (steps, B): a step's targets are one contiguous row (a column of (B, T) cost a strided-copy launch between every two
            # decoder steps -- ~2 us on the serial chain, 12 times)
            start["targets_t"] = start["targets"].t().contiguous()
            if self.training:
                # teacher forcing (models.py:173): every step's next input is known up front -- one gather for the whole
                # sequence, laid out (steps, B, E) so that a step's slice is contiguous, instead of a gather per step
                start["next"] = embedded_text[start["rows"].unsqueeze(0), start["targets"][:, :steps].t()]
            self.multimodal_att_decoder.prepare()          # this step's weight layouts of the decoder's batched GEMMs

        mod_text_audio, mod_text_image, decoder_hidden, decoder_mask = self._encode(
            embedded_text, original_text_lengths, embedded_audio, original_audio_lengths, transformed_images, original_image_lengths,
            decoder_start)
        decoder_cell_state, decoder_input, coverage_vec = start["cell"], start["input"], start["cov"]
        rows, targets, targets_t = start["rows"], start["targets"], start["targets_t"]
        out_distributions, step_losses = [], []
        if self.training:
            next_inputs = start["next"]
        for idx in range(steps):
            tgt = targets_t[idx] if idx < targets_t.size(0) else targets[:, idx]
            # the decoder kernels also emit this step's loss terms: -log(p[target] + 1e-12) (models.py:168-170)
            # and sum(min(att_cov_dist, coverage_vec)) (models.py:177), one value per video
            out_distribution, decoder_hidden, decoder_cell_state, att_cov_dist, coverage_vec, step_loss = \
                self.multimodal_att_decoder.step(decoder_input, decoder_hidden, decoder_cell_state, mod_text_audio,
                                                 mod_text_image, coverage_vec, decoder_mask, target=tgt)
            if self.training:
                decoder_input = next_inputs[idx].unsqueeze(1)                               # models.py:173
            else:
                decoder_input = embedded_text[rows, out_distribution.max(dim=1)[1]].unsqueeze(1)   # models.py:184,:193
            out_distributions.append(out_distribution)
            step_losses.append(step_loss)
        # training adds the coverage loss at every step (models.py:177-178), evaluation once after the loop (:197-198);
        # loss = (sum of the steps' nll + cov_loss_wt * coverage) / steps (models.py:179 / :199)
        cov_loss_wt = 1.0
        loss = Fn.decode_loss(step_losses, steps, cov_loss_wt, self.training)
        return torch.stack(out_distributions).transpose(0, 1), loss

    def summarize(self, text, text_len, audio, audio_len, images, image_len, max_dec_len, targets=None, beam_width=None,
                  no_repeat=False, min_sentences=0, num_samples=None, temperature=1.0, top_k=0, seed=None, top_p=1.0, replacement=True):
        """Extractive summaries of a batch (evaluate.py:107-126, :167-202 with method='greedy'): the eval-mode forward pass with the
        whole greedy decode roll-out on the device, then the greedy sentence selection on the device.  Runs under ``no_grad`` in eval
        mode and gives the caller's ``training`` flag back.  ``targets`` (B, T, 1) or (B, T) with T >= max_dec_len is optional (the
        videos need no labels); with it ``loss`` is the eval loss of ``forward`` (models.py:197-199), else None.
        Returns ``Summary(out_distributions (B, S, M), loss, indices (B, S) int32, counts (B) int32)`` -- the same distributions and
        loss as ``forward`` in eval mode, the same picks as ``decode.get_generated_indices`` (``Summary.to_lists``).
        ``beam_width`` K (1..8) decodes by beam search instead (``MultimodalAttentionDecoder.beam``, one launch): the summary is the
        best hypothesis's -- its indices and counts under the greedy_search rule, its distribution rows as ``out_distributions`` --
        ``loss`` is None and ``beams`` holds every slot (``Beams``).  K = 1 gives the greedy summary.  Not with ``targets``: the eval
        loss is defined by the greedy roll-out.
        ``no_repeat`` (bool) keeps a sentence out of the summary once it is in; ``min_sentences`` (int >= 0) keeps the EOS row from
        ending it before that many sentences (or every sentence of the transcript) are in.  Both constrain the greedy and the beam
        pick, inside the roll-out kernel (the rule at mmb_decoder_greedy_constrained_fused in include/mmbidaf_b200.h); the
        distributions stay the model's.  Not with ``targets``.  With the defaults the launches are exactly the unconstrained ones.
        ``num_samples`` N (1..64) draws N summaries per video instead, in one launch (``MultimodalAttentionDecoder.sample``; the rule
        at mmb_decoder_sample_fused in include/mmbidaf_b200.h): the pick of every step is drawn from p^(1/``temperature``) over the
        candidates -- the ``top_k`` (0: off, else 1..8) likeliest, after the constraints.  ``seed`` None draws the key from the
        device key stream (``ops.rng_next_keys``: fresh samples on every call and graph replay); an int seed reproduces its samples.
        The summary is the likeliest sample's (highest ``Samples.logp``, ties to the lower n); ``samples`` holds all N.  Not with
        ``beam_width`` or ``targets``.  ``top_p`` (in (0, 1], with ``num_samples``) draws each pick from the nucleus, the smallest
        prefix of the candidates (likeliest first) that holds ``top_p`` of their mass, cut from the model's p inside the same launch
        (the rule at mmb_decoder_sample_nucleus_fused in include/mmbidaf_b200.h); 1 is no cut, the same launch as without it.
        ``replacement=False`` (with ``num_samples`` K in 1..8, not with ``top_k`` or ``top_p``) draws K DISTINCT summaries per video, a
        sample without replacement from the tempered, renormalised sequence distribution, by one stochastic beam roll-out
        (``MultimodalAttentionDecoder.beam_sample``; the rule at mmb_decoder_beam_sample_fused in include/mmbidaf_b200.h).
        ``samples`` then holds the K final slots in slot order (``logp`` their scores; an empty slot, when fewer than K sequences
        exist, has an empty summary and logp -inf) and ``inclusion`` (``Inclusion``) their inclusion probabilities and importance
        weights; the summary is the likeliest sample's."""
        from .layers.encoding import length_plan
        from .summarize import Beams, Inclusion, Samples, Summary, best_sample, check_options, sample_logp
        check_options("summarize", targets is not None, beam_width, no_repeat, min_sentences, num_samples, temperature, top_k, seed,
                      top_p, replacement)
        constrained = no_repeat or min_sentences > 0
        was_training = self.training
        self.eval()
        try:
            with torch.no_grad():
                B = text.size(0)
                dec = self.multimodal_att_decoder
                start = {}

                def decoder_start():
                    if targets is not None:
                        start["targets"] = targets.reshape(B, -1).to(text.device).long()
                    dec.prepare()

                enc_a, enc_i, h0, mask = self._encode(text, text_len, audio, audio_len, images, image_len, decoder_start)
                if num_samples is not None:
                    lens = length_plan(text_len, text.device).len_i32
                    key = ops.rng_next_keys(text.device, 1) if seed is None else ops.seed_key(seed, text.device)
                    if not replacement:
                        _, _, scores, rows, phi, keys, paths, slots, kappa = dec.beam_sample(
                            text, h0, enc_a, enc_i, mask, lens, max_dec_len, num_samples, key, temperature, no_repeat, min_sentences)
                        # every final slot's distribution rows: slot path_slots[b, k, s] of step s (zero rows for an empty slot)
                        M = rows.shape[-1]
                        idx = slots.long().clamp_min(0).unsqueeze(3).expand(-1, -1, -1, M)
                        probs = rows.transpose(1, 2).gather(1, idx) * (slots >= 0).unsqueeze(3)
                        samples = Samples(paths, probs, scores[:, -1])
                        sel, cnt = ops.greedy_select(paths.view(B * num_samples, -1), lens.repeat_interleave(num_samples))
                        best_probs, indices, counts = best_sample(samples, sel, cnt)
                        return Summary(best_probs, None, indices, counts, None, samples, Inclusion(phi[:, -1], keys[:, -1], kappa))
                    probs, tokens = dec.sample(text, h0, enc_a, enc_i, mask, lens, max_dec_len, num_samples, key, temperature, top_k,
                                               no_repeat, min_sentences, top_p=top_p)
                    samples = Samples(tokens, probs, sample_logp(probs, tokens, lens))
                    sel, cnt = ops.greedy_select(tokens.view(B * num_samples, -1), lens.repeat_interleave(num_samples))
                    best_probs, indices, counts = best_sample(samples, sel, cnt)
                    return Summary(best_probs, None, indices, counts, None, samples)
                if beam_width is not None:
                    lens = length_plan(text_len, text.device).len_i32
                    tokens, parents, scores, rows, best, path = dec.beam(text, h0, enc_a, enc_i, mask, lens, max_dec_len, beam_width,
                                                                         no_repeat, min_sentences)
                    # the best path's distribution rows: slot path[b, s] of step s
                    M = rows.shape[-1]
                    probs = rows.gather(2, path.long().clamp_min(0)[:, :, None, None].expand(-1, -1, 1, M)).squeeze(2)
                    indices, counts = ops.greedy_select(best, lens)
                    return Summary(probs, None, indices, counts, Beams(tokens, parents, scores, rows))
                if constrained:
                    lens = length_plan(text_len, text.device).len_i32
                    probs, picks, _ = dec.greedy(text, h0, enc_a, enc_i, mask, max_dec_len, text_len=lens, no_repeat=no_repeat,
                                                 min_sentences=min_sentences)
                    indices, counts = ops.greedy_select(picks, lens)
                    return Summary(probs, None, indices, counts)
                probs, argmax, terms = dec.greedy(text, h0, enc_a, enc_i, mask, max_dec_len, target=start.get("targets"))
                # the eval loss exactly as forward forms it: every step's nll, the last step's coverage term, over the steps
                loss = None if terms is None else Fn.decode_loss(list(terms.unbind(0)), max_dec_len, 1.0, False)
                indices, counts = ops.greedy_select(argmax, length_plan(text_len, text.device).len_i32)
        finally:
            self.train(was_training)
        return Summary(probs, loss, indices, counts)

    def score(self, text, text_len, audio, audio_len, images, image_len, max_dec_len, candidates, probs=False):
        """The model's likelihood of given summaries of a batch: every candidate's teacher-forced roll-out of ``max_dec_len`` steps
        (models.py:156-179 in training mode, without dropout), N candidates per video in ONE launch of the cluster kernel
        (``MultimodalAttentionDecoder.force``; the rule at mmb_decoder_forced_fused in include/mmbidaf_b200.h).  Runs like
        :meth:`summarize`: eval mode, ``no_grad``, the encoder half once per video, the caller's ``training`` flag given back.
        ``candidates`` is either a device tensor (B, N, max_dec_len) int64 of token rows with N in 1..64, used as is with every row
        valid (capturable: ``Samples.tokens`` or beam paths go in directly), or host lists, per video, of candidate summaries as
        sentence-index lists, turned into rows by ``summarize.candidate_tokens`` (ValueError, before any device work, for a bad
        candidate).  ``probs`` also returns every step's distribution.  Returns ``Scores(tokens, step_p, logp, loss, valid, probs)``:
        ``logp`` by the rule of ``Samples.logp``, ``loss`` the teacher-forced loss of each row (the training loss of ``forward`` per
        video), -inf / +inf on invalid rows."""
        from .layers.encoding import length_plan
        from .summarize import forced_scores
        if not isinstance(probs, bool):
            raise ValueError(f"score: probs {probs!r}, expected a bool")
        tokens, valid = self._candidate_rows("score", text, text_len, max_dec_len, candidates)
        was_training = self.training
        self.eval()
        try:
            with torch.no_grad():
                dec = self.multimodal_att_decoder
                enc_a, enc_i, h0, mask = self._encode(text, text_len, audio, audio_len, images, image_len, dec.prepare)
                rows, p_tok, terms = dec.force(text, h0, enc_a, enc_i, mask, tokens, want_probs=probs)
                if valid is None:
                    valid = torch.ones(tokens.shape[:2], dtype=torch.bool, device=text.device)
                return forced_scores(tokens, p_tok, terms, valid, length_plan(text_len, text.device).len_i32, rows)
        finally:
            self.train(was_training)

    def sequence_scores(self, text, text_len, audio, audio_len, images, image_len, max_dec_len, candidates):
        """:meth:`score` for training: the same ``Scores`` (``tokens, step_p, logp, loss, valid``; no ``probs``), but in the caller's
        mode and grad mode, as ``forward`` runs -- in training mode the encoders' dropout applies -- and differentiable: ``logp``,
        ``loss`` and ``step_p`` carry gradients to every parameter of the model, so sequence-level objectives (self-critical or
        REINFORCE with sampled candidates, minimum risk, the estimator of a stochastic beam) train it.  With grad enabled the decoder
        runs one forced roll-out that saves every step and one reverse roll-out for the backward
        (``MultimodalAttentionDecoder.force_train``: two launches whatever ``max_dec_len`` is); without, the roll-out of :meth:`score`.
        ``candidates`` as for :meth:`score`: a device tensor (B, N, max_dec_len) int64 with N in 1..64 (capturable), or host lists
        through ``summarize.candidate_tokens``; invalid padding rows get zero gradient.  ValueError, before any device work, for bad
        candidates, and for ``text.requires_grad``: the decoder's next inputs are rows of ``text``, and their gradient is not formed."""
        from .layers.encoding import length_plan
        from .summarize import forced_scores
        if torch.is_tensor(text) and text.requires_grad:
            raise ValueError("sequence_scores: text requires grad; the decoder's next-input rows are gathered from it and their gradient "
                             "is not formed (pass text.detach())")
        tokens, valid = self._candidate_rows("sequence_scores", text, text_len, max_dec_len, candidates)
        if not text.is_cuda:
            raise RuntimeError("mmbidaf_b200 MMBiDAF.sequence_scores runs on a B200 only (no CPU fallback)")
        dec = self.multimodal_att_decoder
        enc_a, enc_i, h0, mask = self._encode(text, text_len, audio, audio_len, images, image_len, dec.prepare)
        if torch.is_grad_enabled():
            p_tok, terms = dec.force_train(text, h0, enc_a, enc_i, mask, tokens)
        else:
            _, p_tok, terms = dec.force(text, h0, enc_a, enc_i, mask, tokens)
        if valid is None:
            valid = torch.ones(tokens.shape[:2], dtype=torch.bool, device=text.device)
        return forced_scores(tokens, p_tok, terms, valid, length_plan(text_len, text.device).len_i32)

    def _candidate_rows(self, who, text, text_len, max_dec_len, candidates):
        """The candidate token rows of :meth:`score` / :meth:`sequence_scores` and their validity (None: every row valid), checked
        before any device work."""
        from .ops import FORCED_MAX_N
        from .summarize import candidate_tokens
        B, S = text.size(0), int(max_dec_len)
        if torch.is_tensor(candidates):
            if candidates.dtype != torch.int64 or candidates.dim() != 3 or candidates.shape[0] != B or \
                    not 1 <= candidates.shape[1] <= FORCED_MAX_N or candidates.shape[2] != S or candidates.device != text.device:
                raise ValueError(f"{who}: candidates {candidates.dtype} {tuple(candidates.shape)} on {candidates.device}, expected "
                                 f"(B={B}, N in 1..{FORCED_MAX_N}, max_dec_len={S}) int64 on {text.device}")
            return candidates, None
        tokens, valid = candidate_tokens(candidates, text_len, S)
        if tokens.shape[0] != B:
            raise ValueError(f"{who}: candidates for {tokens.shape[0]} videos, the batch holds {B}")
        return tokens.to(text.device), valid.to(text.device)

    def _encode(self, embedded_text, original_text_lengths, embedded_audio, original_audio_lengths, transformed_images,
                original_image_lengths, decoder_start):
        """The encoder half of the model (models.py:95-143): embeddings, encoders, masks, both BiDAF blocks, the modality LSTMs and
        the decoder's start state h0.  ``decoder_start()`` is issued on the main stream beside the recurrences (glue that needs no
        encoder output).  Returns (text x audio encoding (B, Lt, 2H), text x image encoding, h0 (B, 1, H), decoder mask (B, M))."""
        B, Lt = embedded_text.size(0), embedded_text.size(1)

        def text_branch():
            emb = self.emb(embedded_text)
            return emb, self.text_enc(emb, original_text_lengths)[0]

        def audio_branch():
            return (self.audio_enc(self.a_emb(embedded_audio), original_audio_lengths)[0],)

        def image_branch():
            img = transformed_images.reshape(-1, *transformed_images.shape[2:])
            feats = self.image_keyframes_emb(img).reshape(B, transformed_images.size(1), -1)
            return feats, self.image_enc(self.i_emb(feats), original_image_lengths)[0]

        masks = {}

        def make_masks():                        # needs only the lengths: issued beside the encoders
            from .layers.encoding import length_plan
            # text mask and decoder mask (the text mask zero-padded to max_transcript_length, models.py:119-123): one launch
            masks["text"], masks["decoder"] = length_plan(original_text_lengths, embedded_text.device).mask(
                Lt, self.max_transcript_length)
            masks["audio"] = self.get_mask(embedded_audio, original_audio_lengths)
            masks["image"] = self.get_mask(transformed_images, original_image_lengths)     # (B, Li, ...): same (B, Li)

        side = {}                                    # made at the end of a chain, on its stream, for the decoder's start

        def audio_aware():
            att = self.bidaf_att_audio(branch["text"], branch["audio"], masks["text"], masks["audio"])
            out = self.mod_t_a(att, original_text_lengths)
            if self.use_streams and out[0].is_cuda:
                side["proj_a"] = self.multimodal_att_decoder.hoist("a", out[0])      # the decoder's hoisted W1 enc_a
                side["hid_a"] = out[1].sum(1)                                        # models.py:143
            return out

        def image_aware():
            att = self.bidaf_att_image(branch["text"], branch["image"], masks["text"], masks["image"])
            out = self.mod_t_i(att, original_text_lengths)
            if self.use_streams and out[0].is_cuda:
                side["proj_i"] = self.multimodal_att_decoder.hoist("i", out[0])      # ... W3 enc_i: this chain ends ~200 us earlier
                side["hid_i"] = out[1].sum(1)
            return out

        branch = {}
        if not (self.use_streams and torch.cuda.is_available()):
            # reference order of the calls (and of the dropout draws): models.py:95-135
            branch["text"] = text_branch()[1]
            branch["audio"] = audio_branch()[0]
            branch["image"] = image_branch()[1]
            make_masks()
            mod_text_audio, text_audio_hidden = audio_aware()
            mod_text_image, text_img_hidden = image_aware()
            decoder_start()
        else:
            # Dependency-driven: the text x image chain (BiDAF + two modality-LSTM layers, ~0.6 ms) needs the text and image encoders
            # only, which finish ~0.3 ms before the 1024-frame audio recurrence -- it runs beside the rest of that recurrence instead of
            # behind a join of all three encoders (which is what two successive fork-joins did: 160 us on the critical path).
            main = torch.cuda.current_stream()
            if getattr(self, "_streams", None) is None or self._streams[0].device != main.device:
                # stream 0 carries the critical path (audio): highest priority, so that its 64 CTAs are never queued behind the others;
                # the text / image chains rank above the weight-gradient lanes (functional.leaf_lanes: default priority), which share the
                # tail of the backward pass with them
                prio = [int(v) for v in os.environ.get("MMB_STREAM_PRIO", "-3,-2,-2").split(",")]
                object.__setattr__(self, "_streams", [torch.cuda.Stream(device=main.device, priority=prio[i]) for i in range(3)])
            s_audio, s_text, s_image = self._streams
            capturing = torch.cuda.is_current_stream_capturing()

            def keep(t, stream):                  # a tensor made on one stream and read on another (no-op inside a graph's pool)
                if not capturing and isinstance(t, torch.Tensor):
                    t.record_stream(stream)

            # every dropout key of the forward pass is drawn on the main stream, in issue order (ops.keys_drawn_on)
            with ops.keys_drawn_on(main):
                for st in self._streams:
                    st.wait_stream(main)
                # The audio chain (embedding -> 1024-step recurrence) is the critical path of the forward pass and the other two encoders
                # have ~250 us of slack: they start when the audio EMBEDDING is done, so that its five small GEMMs / point-wise kernels do not
                # share the chip with theirs (tools/step_timeline.py: 178 us from the start of the step to the start of the audio recurrence
                # with all three chains launched together).
                with torch.cuda.stream(s_audio):
                    audio_emb = self.a_emb(embedded_audio)
                    audio_emb_done = torch.cuda.Event()
                    audio_emb_done.record(s_audio)
                    branch["audio"] = self.audio_enc(audio_emb, original_audio_lengths)[0]
                with torch.cuda.stream(s_text):
                    if self.stagger_encoders:
                        s_text.wait_event(audio_emb_done)
                    branch["text"] = text_branch()[1]
                    text_done = torch.cuda.Event()
                    text_done.record(s_text)
                with torch.cuda.stream(s_image):
                    if self.stagger_encoders:
                        s_image.wait_event(audio_emb_done)
                    branch["image"] = image_branch()[1]
                make_masks()                          # on the main stream, beside the encoders: needs only the lengths
                # ... and so do the keep-masks of the two BiDAF blocks (shapes only): two mask draws less between the audio recurrence and
                # the fused kernel, on the critical path
                d2 = 2 * self.text_enc.rnn.hidden_size
                dev = embedded_text.device
                self.bidaf_att_audio.predraw_dropout((B, Lt, d2), (B, embedded_audio.size(1), d2), dev)
                self.bidaf_att_image.predraw_dropout((B, Lt, d2), (B, transformed_images.size(1), d2), dev)
                for att, st in ((self.bidaf_att_audio, s_audio), (self.bidaf_att_image, s_image)):
                    for t in (getattr(att, "_predrawn", None) or ()):
                        keep(t, st)
                masks_done = torch.cuda.Event()
                masks_done.record(main)
                with torch.cuda.stream(s_image):
                    s_image.wait_event(text_done)
                    s_image.wait_event(masks_done)
                    mod_text_image, text_img_hidden = image_aware()
                with torch.cuda.stream(s_audio):
                    s_audio.wait_event(text_done)
                    s_audio.wait_event(masks_done)
                    mod_text_audio, text_audio_hidden = audio_aware()
                decoder_start()                       # on the main stream, beside the recurrences
                for st in self._streams:
                    main.wait_stream(st)
                keep(branch["text"], s_audio)
                keep(branch["text"], s_image)
                for m in masks.values():
                    keep(m, s_audio)
                    keep(m, s_image)
                for t in (mod_text_audio, text_audio_hidden, mod_text_image, text_img_hidden, branch["text"], branch["audio"], branch["image"],
                          *side.values()):
                    keep(t, main)
        decoder_mask = masks["decoder"]

        # models.py:143-149 (the hidden-state rows are in descending-length order: reference quirk Q3)
        if "hid_a" in side and "hid_i" in side:
            decoder_hidden = (side["hid_a"] + side["hid_i"]).unsqueeze(1)
        else:
            decoder_hidden = (text_audio_hidden.sum(1) + text_img_hidden.sum(1)).unsqueeze(1)
        return mod_text_audio, mod_text_image, decoder_hidden, decoder_mask
