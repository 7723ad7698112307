"""autograd glue: torch.autograd.Function wrappers whose forward AND backward run the library's kernels.

GEMMs that are plain library products (the LSTM input projection x W_ih^T and its transposes in the
backward pass) go through torch.mm / cuBLAS with TF32 off; everything recurrent, soft-maxed or fused is
a hand-written kernel reached through ops.py.
"""
from __future__ import annotations

import contextlib
from typing import Optional, Tuple

import torch

from . import ops


# ---------------------------------------------------------------------------------------------------------------------
# Leaf lanes.  Weight and bias gradients are LEAVES of the backward graph: nothing in the step waits for them except the
# final gradient pack.  Computed inline they sit in stream order between a recurrence and the next op that depends on it
# (tools/step_timeline.py: ~1.2 ms of the 5.9 ms step were such GEMMs and reductions on the critical path, with 84 SMs
# idle beside a 64-CTA recurrence).  Inside ``leaf_lanes()`` every backward below computes what the chain needs (dx) on
# its own stream and hands the leaf products to a side stream; the context joins the lanes on exit.  Outside it (plain
# ``loss.backward()``) everything runs inline as before.
# ---------------------------------------------------------------------------------------------------------------------
class _Lanes:
    # Process-wide on purpose: autograd runs the backward nodes on its own device thread, so the state cannot be thread-local.
    # One training step at a time per process (the design is one process per GPU); a nested / concurrent ``leaf_lanes()`` is
    # a no-op that leaves the products inline.
    enabled = False
    n = 4
    streams = {}          # device index -> [torch.cuda.Stream] * n
    used = set()          # streams that took work since the context was entered
    rr = 0


@contextlib.contextmanager
def leaf_lanes():
    """Run the weight-gradient products of the backward functions in this module on side streams; on exit the CURRENT
    stream waits for them (so the gradients may be consumed right after the ``with`` block).  CUDA-graph capturable."""
    if not torch.cuda.is_available() or _Lanes.enabled:
        yield
        return
    _Lanes.enabled = True
    _Lanes.used = set()
    try:
        yield
    finally:
        _Lanes.enabled = False
        cur = torch.cuda.current_stream()
        for lane in _Lanes.used:
            cur.wait_stream(lane)
        _Lanes.used = set()


@contextlib.contextmanager
def _leaf(*inputs):
    """Everything issued inside runs on a leaf lane, ordered after what the current stream has issued so far.  ``inputs``:
    the tensors read inside that were allocated on other streams (their blocks must not be recycled under the lane)."""
    live = [t for t in inputs if t is not None]
    if not (_Lanes.enabled and live and live[0].is_cuda):
        yield
        return
    cur = torch.cuda.current_stream()
    dev = cur.device.index if cur.device.index is not None else torch.cuda.current_device()
    lanes = _Lanes.streams.get(dev)
    if lanes is None:
        lanes = _Lanes.streams[dev] = [torch.cuda.Stream(device=cur.device) for _ in range(_Lanes.n)]
    lane = lanes[_Lanes.rr % _Lanes.n]
    _Lanes.rr += 1
    _Lanes.used.add(lane)
    lane.wait_stream(cur)
    for t in live:
        t.record_stream(lane)
    with torch.cuda.stream(lane):
        yield


def tall_tn(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a^T b for tall a (N, p), b (N, q) with small p, q -- the shape of every weight gradient here.  As one GEMM that is a
    handful of output tiles looping over K = N on a few CTAs; split into G row blocks it is G times more tiles (a batched
    GEMM) followed by a small sum over the blocks."""
    n, p, q = a.shape[0], a.shape[1], b.shape[1]
    tiles = -(-p // 64) * -(-q // 64)                  # output tiles of a typical 64 x 64 GEMM kernel
    if tiles < 148:                                    # too few to fill the 148 SMs: split the reduction
        for g in (8, 16, 32, 64):                      # fewest row blocks that give ~2 waves of tiles (small partials)
            if n % g == 0 and n // g >= 128 and (tiles * g >= 296 or g == 64):
                return torch.bmm(a.view(g, n // g, p).transpose(1, 2), b.view(g, n // g, q)).sum(dim=0)
    return a.t() @ b


class _TallLinear(torch.autograd.Function):
    """y = x W^T without bias (the Embedding projection, encoding.py:22) whose weight gradient uses :func:`tall_tn`."""

    @staticmethod
    def forward(ctx, x2d, w):
        ctx.save_for_backward(x2d, w)
        return x2d @ w.t()

    @staticmethod
    def backward(ctx, dy):
        x2d, w = ctx.saved_tensors
        dx = dy @ w if ctx.needs_input_grad[0] else None
        with _leaf(dy, x2d):
            dw = tall_tn(dy.contiguous(), x2d)
        return dx, dw


def tall_linear(x: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    shape = x.shape
    return _TallLinear.apply(x.reshape(-1, shape[-1]), weight).view(*shape[:-1], weight.shape[0])


class _TallLinearBias(torch.autograd.Function):
    """y = x W^T + b over tall x (the decoder's hoisted projections W1 enc_a, W3 enc_i, attention.py:152-157): weight and
    bias gradients through :func:`tall_tn` on a leaf lane instead of autograd's inline single GEMM + reduction."""

    @staticmethod
    def forward(ctx, x2d, w, b):
        ctx.save_for_backward(x2d, w)
        return torch.addmm(b, x2d, w.t())

    @staticmethod
    def backward(ctx, dy):
        x2d, w = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dy @ w if ctx.needs_input_grad[0] else None
        with _leaf(dy, x2d):
            dw = tall_tn(dy, x2d)
        with _leaf(dy):
            db = ops.col_sum(dy)
        return dx, dw, db


def tall_linear_bias(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    shape = x.shape
    return _TallLinearBias.apply(x.reshape(-1, shape[-1]), weight, bias).view(*shape[:-1], weight.shape[0])


class _Dropout(torch.autograd.Function):
    """F.dropout on a plain tensor (the embedding inputs, encoding.py:26) with the library's counter-based keep bits: forward and
    backward are the same one-launch kernel with the same key; no mask tensor exists."""

    @staticmethod
    def forward(ctx, x, rng_key, keep_prob):
        ctx.save_for_backward(rng_key)
        ctx.keep_prob = keep_prob
        return ops.dropout_apply(x, rng_key, keep_prob)

    @staticmethod
    def backward(ctx, dy):
        (rng_key,) = ctx.saved_tensors
        return ops.dropout_apply(dy, rng_key, ctx.keep_prob), None, None


def dropout(x: torch.Tensor, drop_prob: float, training: bool) -> torch.Tensor:
    """``F.dropout(x, drop_prob, training)`` as one own launch (fresh key drawn on the device)."""
    if not training or drop_prob <= 0.0:
        return x
    if drop_prob >= 1.0:
        return torch.zeros_like(x)
    return _Dropout.apply(x, ops.rng_next_keys(x.device, 1), 1.0 - float(drop_prob))


def _stacked(parts, shape):
    """``parts`` concatenated along dim 0 and viewed as ``shape``: a VIEW of the first part's storage when the parts are contiguous
    and adjacent in one storage (no launch), else a copy."""
    first = parts[0]
    end = first.storage_offset() + first.numel()
    adjacent = first.is_contiguous()
    for t in parts[1:]:
        adjacent = (adjacent and t.is_contiguous() and t.dtype == first.dtype and t.storage_offset() == end
                    and t.untyped_storage().data_ptr() == first.untyped_storage().data_ptr())
        end += t.numel()
    if adjacent:
        strides, acc = [], 1
        for n in reversed(shape):
            strides.append(acc)
            acc *= n
        return torch.as_strided(first.detach(), shape, tuple(reversed(strides)), first.storage_offset())
    return torch.cat([t.reshape(-1) for t in parts]).view(shape)


class _LstmLayer(torch.autograd.Function):
    """One (bi)directional LSTM layer over padded (B, L, in) with per-sample lengths."""

    @staticmethod
    def forward(ctx, x, lengths, order, rng_key, keep_prob, *weights):
        # weights = (w_ih, w_hh, b_ih, b_hh) per direction; rng_key (device int64 scalar) or None: dropout of the OUTPUT
        # (encoding.py:104 / nn.LSTM's inter-layer dropout) applied inside the recurrence kernels, keep bits hashed from the key
        ndir = len(weights) // 4
        B, L, fan_in = x.shape
        H = weights[1].shape[1]
        # The two directions' weights stacked: views when the parameters already lie side by side in memory (trainer.FlatState puts
        # the forward / reverse tensors of every nn.LSTM layer next to each other for exactly this), else three small copies --
        # five launches per layer in front of the input GEMM, on the serial chain of the step
        w_ih = _stacked([weights[4 * d] for d in range(ndir)], (ndir * 4 * H, fan_in))       # (ndir*4H, in)
        w_hh = _stacked([weights[4 * d + 1] for d in range(ndir)], (ndir, 4 * H, H))         # (ndir, 4H, H)
        b_ih = _stacked([weights[4 * d + 2] for d in range(ndir)], (ndir * 4 * H,))
        b_hh = _stacked([weights[4 * d + 3] for d in range(ndir)], (ndir * 4 * H,))
        bias = b_ih + b_hh
        x2d = x.reshape(B * L, fan_in)
        gates = torch.addmm(bias, x2d, w_ih.t())                                            # plain GEMM (cuBLAS)
        save = any(ctx.needs_input_grad)
        out, h_n, c_n, cell, y = ops.lstm_layer_fwd(gates, w_hh, lengths, order, B, L, H, ndir, save, rng_key, keep_prob)
        if save:
            ctx.save_for_backward(x2d, gates, cell, out, w_ih, w_hh, lengths, order, rng_key)
            ctx.dims = (B, L, H, ndir, fan_in)
            ctx.keep_prob = keep_prob
        ctx.mark_non_differentiable(c_n)
        return (out if y is None else y), h_n, c_n

    @staticmethod
    def backward(ctx, d_out, d_h_n, _d_c_n):
        # the backward kernel overwrites the saved activated gates in place with d(pre-activation) (one buffer, three roles):
        # a second backward over the same graph (retain_graph=True) would read garbage -- refuse it instead
        if getattr(ctx, "consumed", False):
            raise RuntimeError("mmbidaf_b200: the LSTM layer's backward ran twice over one forward (retain_graph=True is not "
                               "supported: its saved gates are overwritten in place)")
        ctx.consumed = True
        x2d, gates, cell, out, w_ih, w_hh, lengths, order, rng_key = ctx.saved_tensors
        B, L, H, ndir, fan_in = ctx.dims
        if d_out is None:
            d_out = torch.zeros_like(out)
        da = ops.lstm_layer_bwd(gates, cell, w_hh, lengths, order, d_out, d_h_n, None, B, L, H, ndir, rng_key, ctx.keep_prob)
        da2d = da.view(B * L, ndir * 4 * H)
        dx = (da2d @ w_ih).view(B, L, fan_in) if ctx.needs_input_grad[0] else None
        # Weight gradients are reductions over all B*L rows with small outputs (4H x in, 4H x H): as ONE GEMM they are a
        # handful of output tiles looping over K = B*L (43 - 100 us each on 14 CTAs).  Batched over the videos instead --
        # sum_b da_b^T x_b -- every video is its own set of tiles (B x more CTAs), and the B partial results are summed
        # by a small reduction.  The recurrent weights take the hidden state that FED step t through shifted views
        # (h[t-1] going forward, h[t+1] going backward; both operands are zero past each length): no concatenation.
        da3 = da.view(B, L, ndir * 4 * H)
        grads = []
        with _leaf(da, x2d):                            # leaves: off the chain that continues with dx, each on its own lane
            dw_ih = tall_tn(da2d, x2d)                                                       # (ndir*4H, in)
        with _leaf(da):
            db = ops.col_sum(da2d)
        for d in range(ndir):
            with _leaf(da, out):
                h_dir = out[:, :, d * H:(d + 1) * H]
                da_dir = da3[:, :, d * 4 * H:(d + 1) * 4 * H]
                if L > 1:
                    lhs, rhs = (da_dir[:, 1:], h_dir[:, :-1]) if d == 0 else (da_dir[:, :-1], h_dir[:, 1:])
                    dw_hh = torch.bmm(lhs.transpose(1, 2), rhs).sum(dim=0)                   # (4H, H)
                else:
                    dw_hh = out.new_zeros(4 * H, H)
            b_d = db[d * 4 * H:(d + 1) * 4 * H]
            grads += [dw_ih[d * 4 * H:(d + 1) * 4 * H], dw_hh, b_d, b_d]
        return (dx, None, None, None, None, *grads)


def lstm_layer(x: torch.Tensor, lengths: torch.Tensor, order: Optional[torch.Tensor], weights,
               rng_key: Optional[torch.Tensor] = None, drop_prob: float = 0.0) -> Tuple[torch.Tensor, torch.Tensor]:
    """x (B,L,in) fp32 CUDA; lengths/order int32 CUDA; weights = [w_ih, w_hh, b_ih, b_hh] * ndir.
    Returns (out (B,L,ndir*H), h_n (B,ndir,H)) in batch order.  With ``rng_key`` (one key of :func:`ops.rng_next_keys`) and
    ``drop_prob`` > 0, ``out`` is dropout(out, drop_prob) applied inside the recurrence kernels (no mask tensor, no extra launch)."""
    if rng_key is None or drop_prob <= 0.0:
        rng_key, keep_prob = None, 1.0
    else:
        keep_prob = 1.0 - float(drop_prob)
    out, h_n, _ = _LstmLayer.apply(x.contiguous(), lengths, order, rng_key, keep_prob, *weights)
    return out, h_n


class _BidafAttention(torch.autograd.Function):
    """Fused BiDAF attention (attention.py:37-75).  Forward = the fused kernels (S never materialised).
    Backward = fused kernels too (S, the soft-maxes and dS are recomputed on chip from the saved soft-max
    statistics): csrc/bidaf_bwd_tc.cu (tcgen05) on the bf16 tier, csrc/bidaf_bwd_f32.cu (FFMA) on the fp32 tier."""

    @staticmethod
    def forward(ctx, text, modality, text_mask, modality_mask, w_text, w_modality, w_cross, bias,
                keep_text, keep_modality, keep_scale, precision):
        save = any(ctx.needs_input_grad)
        res = ops.bidaf_fwd(text, modality, text_mask, modality_mask, w_text, w_modality, w_cross, bias,
                            keep_text, keep_modality, keep_scale, precision, save=save, aux=False)
        if save:
            out, q2c, lse_row, lse_col, bm, ws = res
            ctx.save_for_backward(text, modality, text_mask, modality_mask, w_text, w_modality, w_cross, bias,
                                  keep_text, keep_modality, out, q2c, lse_row, lse_col, bm, ws)
            ctx.keep_scale = keep_scale
            ctx.precision = precision
        return res[0]

    @staticmethod
    def backward(ctx, grad):
        (c, q, c_mask, q_mask, w_c, w_q, w_cq, bias, keep_c, keep_q, out, q2c, lse_row, lse_col, bm, ws) = ctx.saved_tensors
        B, Lc, d = c.shape
        scale = ctx.keep_scale
        dc, dq, dw_c, dw_q, dw_cq, dbias = ops.bidaf_bwd(grad, c, q, c_mask, q_mask, w_c, w_q, w_cq, bias, keep_c, keep_q,
                                                         scale, out, bm, q2c, lse_row, lse_col, ws, ctx.precision)
        return (dc, dq, None, None, dw_c.reshape(w_c.shape), dw_q.reshape(w_q.shape), dw_cq.reshape(w_cq.shape),
                dbias.reshape(bias.shape), None, None, None, None)


def bidaf_attention(text, modality, text_mask, modality_mask, w_text, w_modality, w_cross, bias,
                    keep_text=None, keep_modality=None, keep_scale: float = 1.0, precision: int = ops.PREC_FP32):
    return _BidafAttention.apply(text.contiguous(), modality.contiguous(), text_mask, modality_mask, w_text,
                                 w_modality, w_cross, bias, keep_text, keep_modality, keep_scale, precision)


class _MaskedSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x2d, mask2d, log_mode):
        y = ops.masked_softmax_fwd(x2d, mask2d, log_mode)
        ctx.save_for_backward(y, mask2d)
        ctx.log_mode = log_mode
        return y

    @staticmethod
    def backward(ctx, dy):
        y, mask2d = ctx.saved_tensors
        return ops.masked_softmax_bwd(y, dy, mask2d, ctx.log_mode), None, None


def masked_softmax(logits: torch.Tensor, mask: torch.Tensor, dim: int = -1, log_softmax: bool = False) -> torch.Tensor:
    """attention.py:78-98 for any ``dim``: the axis is moved last, rows go through the CUDA kernel."""
    if not logits.is_cuda:
        raise RuntimeError("mmbidaf_b200 masked_softmax runs on a B200 only (no CPU fallback)")
    dim = dim % logits.dim()
    x = logits.float().movedim(dim, -1)
    m = (mask != 0).expand_as(logits).movedim(dim, -1).contiguous().view(torch.uint8)
    shape = x.shape
    y = _MaskedSoftmax.apply(x.contiguous().view(-1, shape[-1]), m.view(-1, shape[-1]), bool(log_softmax))
    return y.view(shape).movedim(-1, dim)


# ---------------------------------------------------------------------------------------------------------
# Decoder: step kernels under autograd.  Weight gradients are not formed per step: every step's backward
# appends the rows they are built from to a tape, and one set of GEMMs per sequence finishes them.
# ---------------------------------------------------------------------------------------------------------
class DecoderTape:
    """State shared by the steps of one decode sequence (same encoder outputs)."""

    def __init__(self, seq):
        self.seq = seq
        self.rows = {k: [] for k in ("h_prev", "xcat", "h_out", "alpha", "dlog", "da", "dctx12", "dhw4", "dpre", "ctx12")}
        self.d_proj_a = self.d_proj_i = self.vec_acc = self.scal_acc = None
        self._zero = None

    def zero_token(self, like):
        if self._zero is None:
            self._zero = like.new_zeros(1)
        return self._zero

    def open_accumulators(self):
        if self.d_proj_a is None:
            s = self.seq
            self.d_proj_a, self.d_proj_i = torch.zeros_like(s.proj_a), torch.zeros_like(s.proj_i)
            self.vec_acc = s.enc_a.new_zeros(s.B, 6, s.D)
            self.scal_acc = s.enc_a.new_zeros(s.B, 4)


class _DecoderOpen(torch.autograd.Function):
    """Entry of a decode sequence: its backward runs after every step's backward and turns the tape into
    gradients of the encoder outputs, the hoisted projections and the 30 decoder parameters."""

    @staticmethod
    def forward(ctx, tape, proj_a, proj_i, enc_a, enc_i, *params):
        ctx.tape = tape
        ctx.shapes = [p.shape for p in params]
        return enc_a.new_zeros(1)

    @staticmethod
    def backward(ctx, _g):
        tape, r = ctx.tape, ctx.tape.rows
        if getattr(tape, "closed", False):
            raise RuntimeError("mmbidaf_b200: the decoder sequence's backward ran twice over one forward (retain_graph=True is not "
                               "supported: the step tape is consumed and its accumulators are handed out)")
        if not r["dlog"]:
            return (None,) * (5 + len(ctx.shapes))
        tape.closed = True
        s = tape.seq
        B, D, H, E = s.B, s.D, s.H, s.E
        # what the rest of the backward pass waits for first: the gradients of the encoder outputs
        alpha = torch.stack(r["alpha"], dim=0)                               # (S, B, 2, Lt)
        dctx12 = torch.stack(r["dctx12"], dim=0)                             # (S, 2, B, D)
        d_enc_a = torch.bmm(alpha[:, :, 0].permute(1, 2, 0), dctx12[:, 0].permute(1, 0, 2))
        d_enc_i = torch.bmm(alpha[:, :, 1].permute(1, 2, 0), dctx12[:, 1].permute(1, 0, 2))
        with _leaf(tape.vec_acc, tape.scal_acc, *(t for k in ("h_prev", "xcat", "h_out", "dlog", "da", "dhw4", "dpre", "ctx12")
                                                    for t in r[k])):
            grads = _DecoderOpen._param_grads(ctx, tape, r, s)
        for v in r.values():
            v.clear()
        d_proj_a, d_proj_i = tape.d_proj_a, tape.d_proj_i
        tape.d_proj_a = tape.d_proj_i = tape.vec_acc = tape.scal_acc = None      # handed out: never accumulated into again
        return (None, d_proj_a, d_proj_i, d_enc_a, d_enc_i, *grads)

    @staticmethod
    def _param_grads(ctx, tape, r, s):
        B, D = s.B, s.D
        cat = lambda k: torch.cat(r[k], dim=0)
        S = len(r["dlog"])
        kmajor = lambda k: torch.stack(r[k], dim=0).permute(1, 0, 2, 3).reshape(2, S * B, D)   # (S,2,B,D) -> (2,S*B,D)
        return decoder_param_grads(ctx.shapes, s, cat("h_prev"), cat("xcat"), cat("h_out"), cat("dlog"), cat("da"), cat("dhw4"),
                                   kmajor("dpre"), kmajor("ctx12"), tape.vec_acc, tape.scal_acc)


def decoder_param_grads(shapes, s, h_prev, xcat, h_out, dlog, da, dhw4, dpre, ctx12, vec_acc, scal_acc):
    """The gradients of the 30 decoder parameters (``_lib.DECODER_WEIGHT_FIELDS``, reshaped to ``shapes``) from the rows of every step
    of a sequence: h_prev / xcat / h_out (rows, .) the steps' h, [c3 | sent | h] and h', dlog / da / dhw4 (rows, .) their d_logits,
    d_gates and d_hw4, dpre / ctx12 (2, rows, D) d_pre_b and the contexts, vec_acc / scal_acc the kernels' per-row accumulators."""
    D, H, E = s.D, s.H, s.E
    vec, scal = vec_acc.sum(dim=0), scal_acc.sum(dim=0)                  # (6, D), (4)
    d_wh4 = dhw4.t() @ h_prev                                            # (4D, H): W2 | W4 | W_beta_2 | W_beta_4
    hw_sum = dhw4.sum(dim=0)
    d_wb13 = torch.bmm(dpre.transpose(1, 2), ctx12)                      # (2, D, D): W_beta_1 | W_beta_3
    pre_sum = dpre.sum(dim=1)
    d_wcat = da.t() @ xcat                                               # (4H, D+E+H): W_ih | W_hh
    gate_sum = da.sum(dim=0)
    g = {
        "W2": d_wh4[:D], "b2": hw_sum[:D], "Wc1": vec[0].reshape(D, 1), "bc1": hw_sum[:D],
        "v1": vec[2].reshape(1, D), "v1b": scal[0:1],
        "W4": d_wh4[D:2 * D], "b4": hw_sum[D:2 * D], "Wc2": vec[1].reshape(D, 1), "bc2": hw_sum[D:2 * D],
        "v2": vec[3].reshape(1, D), "v2b": scal[1:2],
        "Wb1": d_wb13[0], "bb1": pre_sum[0], "Wb2": d_wh4[2 * D:3 * D], "bb2": hw_sum[2 * D:3 * D],
        "Wb3": d_wb13[1], "bb3": pre_sum[1], "Wb4": d_wh4[3 * D:], "bb4": hw_sum[3 * D:],
        "vb1": vec[4].reshape(1, D), "vb1b": scal[2:3], "vb2": vec[5].reshape(1, D), "vb2b": scal[3:4],
        "lstm_w_ih": d_wcat[:, :D + E], "lstm_w_hh": d_wcat[:, D + E:], "lstm_b_ih": gate_sum, "lstm_b_hh": gate_sum,
        "out_w": dlog.t() @ h_out, "out_b": dlog.sum(dim=0),
    }
    from ._lib import DECODER_WEIGHT_FIELDS
    return [g[name].reshape(shape) for name, shape in zip(DECODER_WEIGHT_FIELDS, shapes)]


class _DecoderStep(torch.autograd.Function):
    """One decoder step.  With ``target`` (B) int64 the kernels also emit the step's loss terms (2,B) and the
    backward pass folds their gradient in (no separate gather / log / min kernels)."""

    @staticmethod
    def forward(ctx, tape, token, sent, h, cell, cov, mask_u8, target):
        probs, h_out, cell_out, att, cov_out, _, saved, lossvec = ops.decoder_step_fwd(
            tape.seq, sent, h, cell, cov, mask_u8, target=target)
        ctx.tape = tape
        ctx.has_token = token is not None
        ctx.fused = target is not None
        extra = (target, att, cov_out) if ctx.fused else ()
        ctx.save_for_backward(h, cell, cov, probs, h_out, cell_out, *saved, *extra)
        ctx.set_materialize_grads(False)
        if lossvec is None:
            lossvec = probs.new_zeros(0)
        return probs, h_out, cell_out, att, cov_out, lossvec

    @staticmethod
    def backward(ctx, d_probs, d_h_out, d_cell_out, d_att, d_cov_out, d_lossvec):
        tape = ctx.tape
        if getattr(tape, "closed", False) or getattr(ctx, "consumed", False):
            raise RuntimeError("mmbidaf_b200: a decoder step's backward ran twice over one forward (retain_graph=True is not supported)")
        ctx.consumed = True
        h, cell, cov, probs, h_out, cell_out, *rest = ctx.saved_tensors
        saved, extra = rest[:7], rest[7:]
        target, att, cov_new = extra if ctx.fused else (None, None, None)
        tape.open_accumulators()
        d_h, d_cell, d_cov, d_logits, d_gates, d_ctx12, d_hw4, d_pre_b = ops.decoder_step_bwd(
            tape.seq, h, cell, cov, probs, cell_out, saved, d_probs, d_h_out, d_cell_out, d_att, d_cov_out,
            tape.d_proj_a, tape.d_proj_i, tape.vec_acc, tape.scal_acc,
            target=target if d_lossvec is not None else None, d_lossvec=d_lossvec, att_cov=att, cov_out=cov_new)
        hw, alpha, beta, ctx12, pb, xcat, gates = saved
        r = tape.rows
        r["h_prev"].append(h); r["xcat"].append(xcat); r["h_out"].append(h_out); r["alpha"].append(alpha)
        r["dlog"].append(d_logits); r["da"].append(d_gates); r["dctx12"].append(d_ctx12); r["dhw4"].append(d_hw4)
        r["dpre"].append(d_pre_b); r["ctx12"].append(ctx12)
        # the token only orders _DecoderOpen.backward after the steps: its gradient is a constant zero (made once per sequence)
        return None, (tape.zero_token(d_h) if ctx.has_token else None), None, d_h, d_cell, d_cov, None, None


class _DecodeLoss(torch.autograd.Function):
    """loss = (sum_s nll_s + w * coverage) / steps from the per-step loss terms (2, B) the decoder kernels emit
    (models.py:168-179 in training: the coverage term of every step; :197-199 in evaluation: of the last step only).
    One stack + one reduction forward and ONE (2, B) tensor shared by every step backward, instead of ~25 one-microsecond
    select / sum / expand kernels between the decoder's forward and backward chains."""

    _coef = {}

    _weights = {}

    @staticmethod
    def forward(ctx, steps, cov_weight, every_step, *terms):
        t = torch.stack(terms)                                           # (S, 2, B)
        S, _, B = t.shape
        ctx.meta = (S, steps, cov_weight, every_step, B)
        # one dot product with a constant weight vector (made once per shape, outside any graph capture: warm-up steps): 1 / steps on
        # every nll term, w / steps on the coverage terms that count -- two launches between the decoder's forward and backward chains
        # instead of seven (stack, three reductions, scale, add, divide)
        key = (t.device, t.dtype, S, steps, cov_weight, every_step, B)
        wvec = _DecodeLoss._weights.get(key)
        if wvec is None:
            w3 = torch.zeros(S, 2, B, dtype=t.dtype)
            w3[:, 0] = 1.0 / steps
            if every_step:
                w3[:, 1] = cov_weight / steps
            else:
                w3[-1, 1] = cov_weight / steps
            wvec = _DecodeLoss._weights[key] = w3.reshape(-1).to(t.device)
        return torch.dot(t.reshape(-1), wvec)

    @staticmethod
    def backward(ctx, g):
        S, steps, w, every_step, B = ctx.meta
        key = (g.device, steps, w, B)
        coef = _DecodeLoss._coef.get(key)
        if coef is None:                                                 # made once (outside any graph capture: warm-up steps)
            coef = _DecodeLoss._coef[key] = torch.tensor([[1.0 / steps], [w / steps]], device=g.device).expand(2, B).contiguous()
        d = coef * g                                                     # (2, B): [d nll | d coverage term], the same for every step
        if every_step:
            return (None, None, None, *([d] * S))
        d_nll_only = torch.stack([d[0], torch.zeros_like(d[0])])
        return (None, None, None, *([d_nll_only] * (S - 1)), d)


def decode_loss(step_losses, steps: int, cov_weight: float, every_step: bool) -> torch.Tensor:
    return _DecodeLoss.apply(steps, cov_weight, every_step, *step_losses)


def decoder_open(tape, proj_a, proj_i, enc_a, enc_i, params):
    return _DecoderOpen.apply(tape, proj_a, proj_i, enc_a, enc_i, *params)


def decoder_step(tape, token, sent, h, cell, cov, mask_u8, target=None):
    return _DecoderStep.apply(tape, token, sent, h, cell, cov, mask_u8, target)


def fold_step_p_grad(g_terms: Optional[torch.Tensor], g_p: Optional[torch.Tensor], p_tok: torch.Tensor) -> torch.Tensor:
    """The loss-term gradient (S, 2, R) the forced roll-out's backward takes, with the gradient of ``p_tok`` (B, N, S) folded into the
    nll coefficient.  p_tok reaches the kernel's backward only through nll = -log(p_tok + 1e-12), whose backward forms
    dp_t = -g_nll / (p_tok + 1e-12): with g_nll -= g_p (p_tok + 1e-12) that is the nll's share plus exactly g_p.  Where p_tok == 0 (a
    masked or out-of-range token) the p_tok gradient is dropped, so the result is never 0 * inf.  Device ops only (capturable)."""
    B, N, S = p_tok.shape
    g = p_tok.new_zeros(S, 2, B * N) if g_terms is None else g_terms.clone(memory_format=torch.contiguous_format)
    if g_p is not None:
        gp, pt = g_p.reshape(B * N, S).t(), p_tok.reshape(B * N, S).t()
        g[:, 0] -= torch.where(pt != 0, gp * (pt + 1e-12), torch.zeros_like(gp))
    return g


class _DecoderForced(torch.autograd.Function):
    """The teacher-forced roll-out of N candidate rows per video under autograd: ONE launch forward
    (ops.decoder_forced_train_fwd), ONE launch backward (ops.decoder_forced_bwd), then the parameter gradients by the GEMMs of
    the per-step path (:func:`decoder_param_grads`) over the S B N rows.  Outputs (p_tok (B,N,S), loss_terms (S,2,B N))."""

    @staticmethod
    def forward(ctx, seq, emb_text, mask_u8, tokens, proj_a, proj_i, enc_a, enc_i, h0, *params):
        p_tok, terms, saved = ops.decoder_forced_train_fwd(seq, emb_text, h0.detach().contiguous(), mask_u8, tokens)
        ctx.seq = seq
        ctx.shapes = [p.shape for p in params]
        ctx.save_for_backward(tokens, p_tok, *saved)
        return p_tok, terms

    @staticmethod
    def backward(ctx, g_p, g_terms):
        # the saved rows are handed out below (d_proj accumulates in place): a second backward would double-count -- refuse it
        if getattr(ctx, "consumed", False):
            raise RuntimeError("mmbidaf_b200: the forced roll-out's backward ran twice over one forward (retain_graph=True is not "
                               "supported)")
        ctx.consumed = True
        seq = ctx.seq
        tokens, p_tok, *saved = ctx.saved_tensors
        B, N, S = tokens.shape
        R, Lt, D, H, E, M = B * N, seq.Lt, seq.D, seq.H, seq.E, seq.M
        g = fold_step_p_grad(g_terms, g_p, p_tok)
        d_proj_a, d_proj_i = torch.zeros_like(seq.proj_a), torch.zeros_like(seq.proj_i)
        vec_acc, scal_acc = seq.enc_a.new_zeros(R, 6, D), seq.enc_a.new_zeros(R, 4)
        d_logits, d_gates, d_hw4, d_ctx12, d_pre_b, d_h0 = ops.decoder_forced_bwd(seq, saved, tokens, g, d_proj_a, d_proj_i,
                                                                                  vec_acc, scal_acc)
        _, _, alpha, _, ctx12, _, xcat, _, _, _, _, h_last = saved
        # d enc_k[b] = sum over (s, n) of alpha_k^T d_ctx12_k: one bmm per modality with K = S N
        d_enc = [torch.bmm(alpha[:, :, k].reshape(S, B, N, Lt).permute(1, 3, 0, 2).reshape(B, Lt, S * N),
                           d_ctx12[:, k].reshape(S, B, N, D).permute(1, 0, 2, 3).reshape(B, S * N, D)) for k in (0, 1)]
        h_in = xcat[:, :, D + E:]                                              # each step's h; step s + 1's is step s's h'
        h_out = torch.cat([h_in[1:], h_last.unsqueeze(0)])
        kmajor = lambda t: t.permute(1, 0, 2, 3).reshape(2, S * R, D)        # (S,2,R,D) -> (2,S*R,D)
        grads = decoder_param_grads(ctx.shapes, seq, h_in.reshape(S * R, H), xcat.reshape(S * R, -1), h_out.reshape(S * R, H),
                                    d_logits.reshape(S * R, M), d_gates.reshape(S * R, 4 * H), d_hw4.reshape(S * R, 4 * D),
                                    kmajor(d_pre_b), kmajor(ctx12), vec_acc, scal_acc)
        return (None, None, None, None, d_proj_a, d_proj_i, d_enc[0], d_enc[1], d_h0.view(B, N, H).sum(1), *grads)


def decoder_forced(seq, emb_text, mask_u8, tokens, proj_a, proj_i, enc_a, enc_i, h0, params):
    """(p_tok (B,N,S), loss_terms (S,2,B N)) of the forced roll-out of ``tokens`` (B,N,S), differentiable in proj_a / proj_i / enc_a /
    enc_i (B,Lt,D), h0 (B,H) and the 30 decoder ``params`` (``_lib.DECODER_WEIGHT_FIELDS`` order)."""
    return _DecoderForced.apply(seq, emb_text, mask_u8, tokens, proj_a, proj_i, enc_a, enc_i, h0, *params)


class _HighwayLayer(torch.autograd.Function):
    """One highway layer: ONE GEMM for gate and transform together + one fused point-wise kernel
    (reference encoding.py:52-59: two GEMMs and seven element-wise kernels per layer)."""

    @staticmethod
    def forward(ctx, x2d, w_gate, b_gate, w_trans, b_trans):
        H = x2d.shape[1]
        w = _stacked([w_gate, w_trans], (2 * H, H))             # (2H, H): views when trainer.FlatState laid them side by side
        pre = torch.addmm(_stacked([b_gate, b_trans], (2 * H,)), x2d, w.t())
        y = ops.highway_fwd(pre, x2d)
        ctx.save_for_backward(x2d, pre, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        x2d, pre, w = ctx.saved_tensors
        H = x2d.shape[1]
        d_pre, dx = ops.highway_bwd(pre, x2d, dy)
        dx = torch.addmm(dx, d_pre, w)                          # direct path + through both linears
        with _leaf(d_pre, x2d):
            dw = tall_tn(d_pre, x2d)                            # (2H, H)
        with _leaf(d_pre):
            db = ops.col_sum(d_pre)
        return dx, dw[:H], db[:H], dw[H:], db[H:]


def highway_layer(x: torch.Tensor, gate: torch.nn.Linear, transform: torch.nn.Linear) -> torch.Tensor:
    shape = x.shape
    y = _HighwayLayer.apply(x.reshape(-1, shape[-1]).contiguous(), gate.weight, gate.bias, transform.weight, transform.bias)
    return y.view(shape)
