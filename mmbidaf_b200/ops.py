"""Thin Python wrappers over the C ABI: allocate outputs with torch, pass raw pointers + stream.

Every function here launches hand-written sm_100a kernels from libmmbidaf_b200.so and raises
if the library or a B200 is missing.  ``launch_count`` counts kernel launches issued through
this module (bench.py reports it as ``gpu_launches``).
"""
from __future__ import annotations

import contextlib
import ctypes
import math
import os
from typing import Optional, Tuple

import torch

from . import _lib

PREC_FP32, PREC_BF16 = 0, 1
launch_count = 0


def _count(n: int) -> None:
    global launch_count
    launch_count += n


def _u8(mask: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if mask is None:
        return None
    if mask.dtype == torch.bool:
        return mask.contiguous().view(torch.uint8)
    return mask.to(torch.uint8).contiguous()


def bidaf_fwd(text: torch.Tensor, modality: torch.Tensor, text_mask: torch.Tensor, modality_mask: torch.Tensor,
              w_text: torch.Tensor, w_modality: torch.Tensor, w_cross: torch.Tensor, bias: torch.Tensor,
              keep_text: Optional[torch.Tensor] = None, keep_modality: Optional[torch.Tensor] = None,
              keep_scale: float = 1.0, precision: int = PREC_FP32, save: bool = False, aux: bool = True):
    """Fused BiDAF forward (attention.py:37-75).  Returns (out (B,Lc,4d), q2c (B,Lq,d), lse_row (B,Lc),
    lse_col (B,Lq)); with ``save`` also (bm (B,Lc,d), workspace) -- everything the backward pass needs.  ``aux=False`` (bf16 tier,
    no ``save``): only ``out`` is computed and written (inference: the reference's forward returns nothing else);
    the other three results are None."""
    L = _lib.lib()
    assert text.dtype == torch.float32 and modality.dtype == torch.float32
    B, Lc, d = text.shape
    Lq = modality.shape[1]
    text, modality = text.contiguous(), modality.contiguous()
    tm, mm = _u8(text_mask.reshape(B, Lc)), _u8(modality_mask.reshape(B, Lq))
    kt, km = _u8(keep_text), _u8(keep_modality)
    wt, wm, wc = (w.detach().reshape(-1).contiguous() for w in (w_text, w_modality, w_cross))
    out = torch.empty(B, Lc, 4 * d, device=text.device, dtype=torch.float32)
    want_aux = aux or save or precision != PREC_BF16
    q2c = torch.empty(B, Lq, d, device=text.device, dtype=torch.float32) if want_aux else None
    bm = torch.empty(B, Lc, d, device=text.device, dtype=torch.float32) if save else None
    lse_row = torch.empty(B, Lc, device=text.device, dtype=torch.float32) if want_aux else None
    lse_col = torch.empty(B, Lq, device=text.device, dtype=torch.float32) if want_aux else None
    p = _lib.ptr
    ws_bytes = L.mmb_bidaf_workspace_bytes(B, Lc, Lq, d, int(precision), int(km is not None))
    ws = torch.empty(ws_bytes, device=text.device, dtype=torch.uint8) if ws_bytes else None
    _lib.check(L.mmb_bidaf_fwd(p(text), p(modality), p(tm), p(mm), p(wt), p(wm), p(wc), p(bias.detach().contiguous()),
                               p(kt), p(km), float(keep_scale), p(out), p(q2c), p(bm), p(lse_row), p(lse_col), p(ws),
                               B, Lc, Lq, d, int(precision), _lib.stream()), "mmb_bidaf_fwd")
    _count(2)          # fp32: two pass launches; bf16: pack + one fused tensor-core launch
    if save:
        return out, q2c, lse_row, lse_col, bm, ws
    return out, q2c, lse_row, lse_col


def bidaf_bwd(grad_out: torch.Tensor, text: torch.Tensor, modality: torch.Tensor, text_mask: torch.Tensor,
              modality_mask: torch.Tensor, w_text: torch.Tensor,
              w_modality: torch.Tensor, w_cross: torch.Tensor, bias: torch.Tensor, keep_text: Optional[torch.Tensor],
              keep_modality: Optional[torch.Tensor], keep_scale: float, out: torch.Tensor, bm: torch.Tensor,
              q2c: torch.Tensor, lse_row: torch.Tensor, lse_col: torch.Tensor, fwd_ws: Optional[torch.Tensor],
              precision: int):
    """Fused BiDAF backward (the autograd gradient of attention.py:37-75) from what :func:`bidaf_fwd` saved.
    Returns (d_text, d_modality, d_w_text (d), d_w_modality (d), d_w_cross (d), d_bias (1))."""
    L = _lib.lib()
    B, Lc, d = text.shape
    Lq = modality.shape[1]
    dev = text.device
    kt, km = _u8(keep_text), _u8(keep_modality)
    tm, mm = _u8(text_mask.reshape(B, Lc)), _u8(modality_mask.reshape(B, Lq))
    wt, wm, wc = (w.detach().reshape(-1).contiguous() for w in (w_text, w_modality, w_cross))
    d_text = torch.empty_like(text)
    d_modality = torch.empty_like(modality)
    d_w = torch.empty(3, d, device=dev, dtype=torch.float32)
    d_bias = torch.empty(1, device=dev, dtype=torch.float32)
    ws_bytes = L.mmb_bidaf_bwd_workspace_bytes(B, Lc, Lq, d, int(precision))
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8) if ws_bytes else None
    p = _lib.ptr
    _lib.check(L.mmb_bidaf_bwd(p(grad_out.contiguous()), p(text), p(modality), p(tm), p(mm), p(wt), p(wm), p(wc),
                               p(bias.detach().contiguous()), p(kt), p(km), float(keep_scale), p(out), p(bm), p(q2c),
                               p(lse_row), p(lse_col), p(fwd_ws), p(ws), p(d_text), p(d_modality), p(d_w[0]), p(d_w[1]),
                               p(d_w[2]), p(d_bias), B, Lc, Lq, d, int(precision), _lib.stream()), "mmb_bidaf_bwd")
    _count(3 if precision == PREC_BF16 else 5)
    if precision == PREC_BF16 and os.environ.get("MMB_BIDAF_BWD_TRACE"):      # debugging aid: clock stamps at the end of the workspace
        bidaf_bwd.last_trace = ws[-3 * 256 * 8:].view(torch.int64).view(3, 256)
    return d_text, d_modality, d_w[0], d_w[1], d_w[2], d_bias


def lstm_layer_fwd(gates: torch.Tensor, w_hh: torch.Tensor, lengths: torch.Tensor, order: Optional[torch.Tensor],
                   B: int, L: int, H: int, ndir: int, save: bool, rng_key: Optional[torch.Tensor] = None, keep_prob: float = 1.0):
    """Persistent LSTM recurrence of one layer (encoding.py:96).  ``gates`` (B,L,ndir,4H) holds the input
    projection on entry and, when ``save``, the activated gates on exit.  Returns (out (B,L,ndir*H),
    h_n (B,ndir,H), c_n (B,ndir,H), cell (B,L,ndir,H) or None, y): with ``rng_key`` (a device int64 scalar from :func:`rng_next_keys`)
    the kernel also writes ``y`` = dropout(out, 1 - keep_prob) (encoding.py:104 / nn.LSTM's inter-layer dropout); else ``y`` is None."""
    lib = _lib.lib()
    assert gates.dtype == torch.float32 and gates.numel() == B * L * ndir * 4 * H
    assert lengths.dtype == torch.int32 and (order is None or order.dtype == torch.int32)
    dev = gates.device
    out = torch.empty(B, L, ndir * H, device=dev, dtype=torch.float32)
    h_n = torch.empty(B, ndir, H, device=dev, dtype=torch.float32)
    c_n = torch.empty(B, ndir, H, device=dev, dtype=torch.float32)
    cell = torch.empty(B, L, ndir, H, device=dev, dtype=torch.float32) if save else None
    p = _lib.ptr
    if rng_key is None:
        _lib.check(lib.mmb_bilstm_fwd(p(gates), p(w_hh), p(lengths), p(order), p(out), p(h_n), p(c_n), p(cell),
                                      B, L, H, ndir, int(save), _lib.stream()), "mmb_bilstm_fwd")
        y = None
    else:
        assert rng_key.dtype == torch.int64 and rng_key.is_cuda
        y = torch.empty_like(out)
        _lib.check(lib.mmb_bilstm_fwd_dropout(p(gates), p(w_hh), p(lengths), p(order), p(out), p(y), p(h_n), p(c_n), p(cell),
                                              p(rng_key), float(keep_prob), B, L, H, ndir, int(save), _lib.stream()),
                   "mmb_bilstm_fwd_dropout")
    _count(1)
    return out, h_n, c_n, cell, y


def lstm_layer_bwd(gates: torch.Tensor, cell: torch.Tensor, w_hh: torch.Tensor, lengths: torch.Tensor,
                   order: Optional[torch.Tensor], dout: torch.Tensor, dh_n: Optional[torch.Tensor],
                   dc_n: Optional[torch.Tensor], B: int, L: int, H: int, ndir: int, rng_key: Optional[torch.Tensor] = None,
                   keep_prob: float = 1.0) -> torch.Tensor:
    """BPTT of :func:`lstm_layer_fwd`; overwrites ``gates`` with d(pre-activation) and returns it.  With ``rng_key``, ``dout`` is
    the gradient of the DROPPED output ``y``."""
    lib = _lib.lib()
    p = _lib.ptr
    dh = None if dh_n is None else dh_n.contiguous()
    dc = None if dc_n is None else dc_n.contiguous()
    if rng_key is None:
        _lib.check(lib.mmb_bilstm_bwd(p(gates), p(cell), p(w_hh), p(lengths), p(order), p(dout.contiguous()), p(dh), p(dc),
                                      B, L, H, ndir, _lib.stream()), "mmb_bilstm_bwd")
    else:
        _lib.check(lib.mmb_bilstm_bwd_dropout(p(gates), p(cell), p(w_hh), p(lengths), p(order), p(dout.contiguous()), p(dh), p(dc),
                                              p(rng_key), float(keep_prob), B, L, H, ndir, _lib.stream()), "mmb_bilstm_bwd_dropout")
    _count(1)
    return gates


_rng_state = {}


_rng_seed_override = {"seed": None}


def rng_seed(seed: int, device=None) -> None:
    """(Re)seed the device-resident key stream of the in-kernel dropout (all devices, or one); states created later start from it too."""
    _rng_seed_override["seed"] = int(seed)
    for dev, st in _rng_state.items():
        if device is None or dev == torch.device(device):
            st.fill_(int(seed) & 0x7FFFFFFFFFFFFFFF)


_key_stream = {"stream": None}


@contextlib.contextmanager
def keys_drawn_on(stream: torch.cuda.Stream):
    """Inside, :func:`rng_next_keys` draws on ``stream`` whatever the current stream is, and the current stream waits for the keys.
    The key state is one device word that every draw reads and advances: draws issued from concurrent streams would advance it
    in whatever order the GPU runs them, so which layer gets which key (and whether two get the same one) would change from run to
    run.  On one stream the draws run in the order they are issued."""
    saved, _key_stream["stream"] = _key_stream["stream"], stream
    try:
        yield
    finally:
        _key_stream["stream"] = saved


def rng_next_keys(device, n: int) -> torch.Tensor:
    """``n`` fresh dropout keys (int64, on ``device``), drawn ON the device from a resident state: one tiny launch, capturable (a graph
    replay draws new keys).  The state is seeded from torch's seed at first use."""
    device = torch.device(device)
    cur = torch.cuda.current_stream(device)
    draw = _key_stream["stream"] if _key_stream["stream"] is not None and _key_stream["stream"].device == cur.device else cur
    with torch.cuda.stream(draw):
        st = _rng_state.get(device)
        if st is None:
            if torch.cuda.is_current_stream_capturing():
                # created inside a capture, the state's initial fill would be replayed too: the same masks on every replay
                raise RuntimeError("mmbidaf_b200: the dropout key state must exist before a CUDA-graph capture (run one eager step, as "
                                   "Trainer.capture does, or call ops.rng_next_keys once)")
            # (every rank of a data-parallel job draws its own masks: the rank is mixed into the seed)
            import torch.distributed as dist
            rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
            st = _rng_state[device] = torch.full((1,), (((torch.initial_seed() if _rng_seed_override["seed"] is None else _rng_seed_override["seed"]) + 0x51ED27 * rank)
                                                  * 0x9E3779B97F4A7C15 + 0x1234567)
                                                 & 0x7FFFFFFFFFFFFFFF, dtype=torch.int64, device=device)
        keys = torch.empty(n, dtype=torch.int64, device=device)
        _lib.check(_lib.lib().mmb_rng_next(_lib.ptr(st), _lib.ptr(keys), n, _lib.stream()), "mmb_rng_next")
    _count(1)
    if draw != cur:
        cur.wait_stream(draw)
        if not torch.cuda.is_current_stream_capturing():
            keys.record_stream(cur)                      # allocated on the draw stream, read on this one
    return keys


def dropout_mask_u8(rng_key: torch.Tensor, keep_prob: float, shape) -> torch.Tensor:
    """The keep bits of ``rng_key`` for a tensor of ``shape`` as bytes (uint8 0 / 1): what the BiDAF kernels take as ``keep_text`` /
    ``keep_modality`` (attention.py:66-67) -- one own launch instead of ATen's bernoulli_."""
    n = 1
    for d in shape:
        n *= int(d)
    mask = torch.empty(n, dtype=torch.uint8, device=rng_key.device)
    _lib.check(_lib.lib().mmb_dropout_mask(_lib.ptr(rng_key), float(keep_prob), n, _lib.ptr(mask), _lib.stream()), "mmb_dropout_mask")
    _count(1)
    return mask.view(*shape)


def dropout_mask(rng_key: torch.Tensor, keep_prob: float, shape) -> torch.Tensor:
    """The keep mask (bool, ``shape``) the kernels derive from ``rng_key`` for a tensor of that shape (tests / debugging)."""
    return dropout_mask_u8(rng_key, keep_prob, shape).bool()


def dropout_apply(x: torch.Tensor, rng_key: torch.Tensor, keep_prob: float) -> torch.Tensor:
    """dropout(x, 1 - keep_prob) with the keep bits of ``rng_key`` (encoding.py:26): one launch, no mask tensor."""
    assert x.dtype == torch.float32 and x.is_cuda and rng_key.dtype == torch.int64
    x = x.contiguous()
    y = torch.empty_like(x)
    _lib.check(_lib.lib().mmb_dropout_apply(_lib.ptr(x), _lib.ptr(y), _lib.ptr(rng_key), float(keep_prob), x.numel(), _lib.stream()),
               "mmb_dropout_apply")
    _count(1)
    return y


class DecoderWeights:
    """The decoder's weights laid out for the batched GEMMs and kernels of a step (attention.py:110-143 parameters).
    Depends on the parameters only, so it can be built beside the encoders (MMBiDAF.forward) instead of in front of the
    first decoder step.  ``params`` maps the names of ``_lib.DECODER_WEIGHT_FIELDS`` to parameter tensors."""

    def __init__(self, params: dict, out_size: int):
        P = {k: v.detach() for k, v in params.items()}
        self.D, self.H = P["W2"].shape
        self.M = out_size
        self.E = P["lstm_w_ih"].shape[1] - self.D
        self.Wh4 = torch.cat([P["W2"], P["W4"], P["Wb2"], P["Wb4"]], dim=0).contiguous()           # (4D, H)
        # every bias that ends up inside the same tanh is added once, with the h projection: W2 h + b2 + bc1 (attention.py:147),
        # W_beta_2 h + bb2 + bb1 (the bias of W_beta_1 c_1, :161) -- so the c_k projection below is a bias-free GEMM
        self.bh4 = torch.cat([P["b2"] + P["bc1"], P["b4"] + P["bc2"], P["bb2"] + P["bb1"], P["bb4"] + P["bb3"]]).contiguous()
        self.Wb13 = torch.stack([P["Wb1"], P["Wb3"]]).contiguous()                                 # (2, D, D)
        self.Wcat = torch.cat([P["lstm_w_ih"], P["lstm_w_hh"]], dim=1).contiguous()                # (4H, D+E+H)
        # backward: d ctx = d_gates W_ih[:, :D]; d h = [d_gates | d_hw4] [W_hh ; Wh4] (one GEMM over the stacked gradients)
        self.Wcat_ctx = P["lstm_w_ih"][:, :self.D].contiguous()                                    # (4H, D)
        self.Wh_stack = torch.cat([P["lstm_w_hh"], self.Wh4], dim=0).contiguous()                   # (4H + 4D, H)
        self.bcat = (P["lstm_b_ih"] + P["lstm_b_hh"]).contiguous()
        self.out_w, self.out_b = P["out_w"].contiguous(), P["out_b"].contiguous()
        # transposed copies for the one-kernel step (csrc/decoder_fused.cu): consecutive threads read consecutive output neurons
        self.Wh4t, self.Wcatt, self.out_wt = self.Wh4.t().contiguous(), self.Wcat.t().contiguous(), self.out_w.t().contiguous()
        self.Wb13t = self.Wb13.transpose(1, 2).contiguous()
        # backward: d h = d_logits out.weight with K = M padded to a multiple of 8 (M = 409 is odd: an un-aligned GEMM otherwise)
        self.Mp = (self.M + 7) // 8 * 8
        self.out_w_pad = torch.cat([self.out_w, self.out_w.new_zeros(self.Mp - self.M, self.H)], dim=0).contiguous()
        flat = lambda k: P[k].reshape(-1).contiguous()
        self.v1, self.wc1, self.v2, self.wc2 = flat("v1"), flat("Wc1"), flat("v2"), flat("Wc2")
        self.vb1, self.vb2 = flat("vb1"), flat("vb2")
        self.v1b, self.v2b, self.vb1b, self.vb2b = flat("v1b"), flat("v2b"), flat("vb1b"), flat("vb2b")


class DecoderSeq:
    """Everything that is constant over the steps of one decode sequence (attention.py:145-186): the weight layouts
    (:class:`DecoderWeights`, built here unless handed in), the hoisted projections and the chunking."""

    def __init__(self, params: dict, enc_a, enc_i, proj_a, proj_i, out_size: int, weights: Optional[DecoderWeights] = None):
        w = weights if weights is not None else DecoderWeights(params, out_size)
        self.__dict__.update(w.__dict__)
        self.enc_a, self.enc_i = enc_a.detach().contiguous(), enc_i.detach().contiguous()
        self.proj_a, self.proj_i = proj_a.detach().contiguous(), proj_i.detach().contiguous()
        self.B, self.Lt, D = self.enc_a.shape
        if D != self.D or out_size != self.M:
            raise RuntimeError(f"DecoderSeq: encoder width {D} / output size {out_size} do not match the weights ({self.D}, {self.M})")
        self.nch = _lib.lib().mmb_decoder_chunks(self.B, self.Lt)
        # per-video arrival counters of the chunk-parallel kernels (zero between launches): one set per direction
        self.counters = torch.zeros(2, self.B, device=self.enc_a.device, dtype=torch.int32)


def decoder_cut(B: int, Lt: int) -> str:
    """Which cut of the decoder step runs for B videos of Lt text rows: "fused" (one cluster kernel per step, or the whole greedy
    roll-out in one launch) or "chunks" (the five-kernel chunk-parallel cut); MMB_DECODER_CUT overrides ("head" is a backward-only
    cross-check; the forward treats anything but "chunks" as "fused")."""
    cut = os.environ.get("MMB_DECODER_CUT")
    if cut is None:
        # a cluster (4 or 8 CTAs) per video: at most ~1000 CTAs worth of text rows per launch keeps every CTA's share of the text sweep
        # short; long lectures (config 5: 16 x 4096 rows) are better spread over the (chunks x B) grid of the five-kernel cut
        cut = "fused" if B * Lt <= 20000 else "chunks"
    return cut


def decoder_step_fwd(seq: DecoderSeq, sent, h, cell, coverage, mask_u8, want_argmax: bool = False, target=None):
    """One decoder step.  sent (B,E), h/cell (B,H), coverage (B,Lt), mask_u8 (B,M) uint8 -- contiguous fp32 CUDA.
    With ``target`` (B) int64 the kernels also emit the step's loss terms ``lossvec`` (B,2) =
    [-log(p[target]+1e-12), sum_t min(att_cov, coverage')] (models.py:168-178).
    Returns (probs, h', cell', att_cov, coverage', argmax|None, saved, lossvec|None) where ``saved`` is what
    :func:`decoder_step_bwd` needs: (hw, alpha, beta, ctx12, pb, xcat, gates)."""
    lib = _lib.lib()
    B, Lt, D, H, E, M, nch = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M, seq.nch
    f32 = dict(device=h.device, dtype=torch.float32)
    p = _lib.ptr
    st = _lib.stream()
    cut = decoder_cut(B, Lt)
    if cut != "chunks":
        # the whole step as one cluster kernel (csrc/decoder_fused.cu); MMB_DECODER_CUT=chunks forces the five-kernel cut below
        hw, alpha, beta = torch.empty(B, 4 * D, **f32), torch.empty(B, 2, Lt, **f32), torch.empty(B, 2, **f32)
        ctx12, pb = torch.empty(2, B, D, **f32), torch.empty(2, B, D, **f32)
        xcat, gates = torch.empty(B, D + E + H, **f32), torch.empty(B, 4 * H, **f32)
        probs, h_out, cell_out = torch.empty(B, M, **f32), torch.empty(B, H, **f32), torch.empty(B, H, **f32)
        att_cov, cov_out = torch.empty(B, Lt, **f32), torch.empty(B, Lt, **f32)
        argmax = torch.empty(B, device=h.device, dtype=torch.int64) if want_argmax else None
        lossvec = torch.empty(2, B, **f32) if target is not None else None       # [nll | coverage term]
        _lib.check(lib.mmb_decoder_step_fused_fwd(
            p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(seq.Wh4t), p(seq.bh4), p(seq.v1), p(seq.wc1), p(seq.v2),
            p(seq.wc2), p(seq.v1b), p(seq.v2b), p(seq.Wb13t), p(seq.vb1), p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(seq.Wcatt),
            p(seq.bcat), p(seq.out_wt), p(seq.out_b), p(sent), p(h), p(cell), p(coverage), p(mask_u8), p(target), p(probs), p(h_out),
            p(cell_out), p(att_cov), p(cov_out), p(argmax), p(None if lossvec is None else lossvec[0]),
            p(None if lossvec is None else lossvec[1]), p(hw), p(alpha), p(beta), p(ctx12), p(pb), p(xcat), p(gates),
            B, Lt, D, H, E, M, st), "mmb_decoder_step_fused_fwd")
        _count(1)
        return probs, h_out, cell_out, att_cov, cov_out, argmax, (hw, alpha, beta, ctx12, pb, xcat, gates), lossvec
    hw = torch.addmm(seq.bh4, h, seq.Wh4.t())                                  # (B, 4D)  library GEMM
    alpha = torch.empty(B, 2, Lt, **f32)
    stats, ctxp = torch.empty(B, nch, 4, **f32), torch.empty(B, nch, 2, D, **f32)
    ctx12, scale = torch.empty(2, B, D, **f32), torch.empty(B, 2, nch, **f32)
    _lib.check(lib.mmb_decoder_attn_fwd(p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(hw), p(coverage),
                                        p(seq.v1), p(seq.wc1), p(seq.v2), p(seq.wc2), p(seq.v1b), p(seq.v2b), p(alpha),
                                        p(stats), p(ctxp), p(ctx12), p(scale), p(seq.counters[0]), B, Lt, D, nch, st),
               "mmb_decoder_attn_fwd")
    pb = torch.bmm(ctx12, seq.Wb13.transpose(1, 2))                            # (2, B, D)  library GEMM (bias: see DecoderSeq)
    xcat = torch.empty(B, D + E + H, **f32)
    att_cov, cov_out, beta = torch.empty(B, Lt, **f32), torch.empty(B, Lt, **f32), torch.empty(B, 2, **f32)
    lossvec = torch.empty(2, B, **f32) if target is not None else None       # [nll | coverage term]
    _lib.check(lib.mmb_decoder_attn_finish(p(pb), p(hw), p(ctx12), p(scale), p(coverage), p(sent), p(h), p(seq.vb1),
                                           p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(alpha), p(xcat), p(att_cov),
                                           p(cov_out), p(beta), p(None if lossvec is None else lossvec[1]),
                                           B, Lt, D, E, H, nch, st), "mmb_decoder_attn_finish")
    gates = torch.addmm(seq.bcat, xcat, seq.Wcat.t())                          # (B, 4H)  library GEMM
    h_out, cell_out = torch.empty(B, H, **f32), torch.empty(B, H, **f32)
    _lib.check(lib.mmb_decoder_cell_fwd(p(gates), p(cell), p(h_out), p(cell_out), B, H, st), "mmb_decoder_cell_fwd")
    probs = torch.addmm(seq.out_b, h_out, seq.out_w.t())                       # (B, M) logits, library GEMM
    argmax = torch.empty(B, device=h.device, dtype=torch.int64) if want_argmax else None
    _lib.check(lib.mmb_decoder_out_softmax(p(probs), p(mask_u8), p(argmax), p(target),
                                           p(None if lossvec is None else lossvec[0]), B, M, st), "mmb_decoder_out_softmax")
    _count(5)
    return probs, h_out, cell_out, att_cov, cov_out, argmax, (hw, alpha, beta, ctx12, pb, xcat, gates), lossvec


def decoder_greedy_fwd(seq: DecoderSeq, emb_text, h0, mask_u8, steps: int, target=None):
    """The greedy roll-out of ``steps`` decoder steps in eval mode as ONE launch (csrc/decoder_fused.cu, models.py:156-199).
    emb_text (B,Lt,E) fp32, h0 (B,H) fp32, mask_u8 (B,M) uint8, target (B,T) int64 with T >= steps or None.
    Returns (probs (B,steps,M), argmax (B,steps) int64, loss_terms (steps,2,B) = per step [nll | coverage term] or None)."""
    lib = _lib.lib()
    B, Lt, D, H, E, M = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M
    dev = h0.device
    if emb_text.shape != (B, Lt, E) or h0.shape != (B, H) or mask_u8.shape != (B, M):
        raise ValueError(f"decoder_greedy_fwd: emb_text {tuple(emb_text.shape)}, h0 {tuple(h0.shape)}, mask {tuple(mask_u8.shape)} "
                         f"for B={B} Lt={Lt} E={E} H={H} M={M}")
    T = 0
    if target is not None:
        T = target.shape[1]
        if target.dtype != torch.int64 or target.shape[0] != B or T < steps:
            raise ValueError(f"decoder_greedy_fwd: target {tuple(target.shape)} {target.dtype} for B={B}, {steps} steps")
    probs = torch.empty(B, steps, M, device=dev, dtype=torch.float32)
    argmax = torch.empty(B, steps, device=dev, dtype=torch.int64)
    terms = torch.empty(steps, 2, B, device=dev, dtype=torch.float32) if target is not None else None
    p = _lib.ptr
    _lib.check(lib.mmb_decoder_greedy_fused(
        p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(seq.Wh4t), p(seq.bh4), p(seq.v1), p(seq.wc1), p(seq.v2),
        p(seq.wc2), p(seq.v1b), p(seq.v2b), p(seq.Wb13t), p(seq.vb1), p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(seq.Wcatt),
        p(seq.bcat), p(seq.out_wt), p(seq.out_b), p(emb_text), p(h0), p(mask_u8), p(target), p(probs), p(argmax), p(terms),
        B, Lt, D, H, E, M, int(steps), int(T), _lib.stream()), "mmb_decoder_greedy_fused")
    _count(1)
    return probs, argmax, terms


def _check_constraints(who: str, no_repeat, min_sentences) -> None:
    if not isinstance(no_repeat, int) or no_repeat not in (0, 1):
        raise ValueError(f"{who}: no_repeat {no_repeat!r}, expected a bool")
    if isinstance(min_sentences, bool) or not isinstance(min_sentences, int) or min_sentences < 0:
        raise ValueError(f"{who}: min_sentences {min_sentences!r}, expected an int >= 0")


def decoder_greedy_constrained_fwd(seq: DecoderSeq, emb_text, h0, mask_u8, text_len_i32, steps: int, no_repeat: bool = False,
                                   min_sentences: int = 0):
    """The constrained greedy roll-out (rule at mmb_decoder_greedy_constrained_fused in include/mmbidaf_b200.h) as ONE launch of the
    cluster kernel, whatever ``decoder_cut`` says: there is no chunk-cut constrained greedy.  ``no_repeat`` blocks a sentence once
    picked; the EOS row is not picked before ``min_sentences`` sentences (or every sentence) are in.  Inputs as
    :func:`decoder_greedy_fwd` without a target, plus text_len_i32 (B) int32 (the EOS row of video b is text_len[b] - 1).
    Returns (probs (B,steps,M), picks (B,steps) int64) -- the distributions are the unconstrained model's, bit for bit."""
    lib = _lib.lib()
    B, Lt, D, H, E, M = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M
    dev = h0.device
    _check_constraints("decoder_greedy_constrained_fwd", no_repeat, min_sentences)
    if int(steps) <= 0:
        raise ValueError(f"decoder_greedy_constrained_fwd: {steps} steps")
    if emb_text.shape != (B, Lt, E) or h0.shape != (B, H) or mask_u8.shape != (B, M) or text_len_i32.shape != (B,):
        raise ValueError(f"decoder_greedy_constrained_fwd: emb_text {tuple(emb_text.shape)}, h0 {tuple(h0.shape)}, "
                         f"mask {tuple(mask_u8.shape)}, text_len {tuple(text_len_i32.shape)} for B={B} Lt={Lt} E={E} H={H} M={M}")
    if text_len_i32.dtype != torch.int32:
        raise ValueError(f"decoder_greedy_constrained_fwd: text_len {text_len_i32.dtype}, not int32")
    S = int(steps)
    probs = torch.empty(B, S, M, device=dev, dtype=torch.float32)
    picks = torch.empty(B, S, device=dev, dtype=torch.int64)
    p = _lib.ptr
    _lib.check(lib.mmb_decoder_greedy_constrained_fused(
        p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(seq.Wh4t), p(seq.bh4), p(seq.v1), p(seq.wc1), p(seq.v2),
        p(seq.wc2), p(seq.v1b), p(seq.v2b), p(seq.Wb13t), p(seq.vb1), p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(seq.Wcatt),
        p(seq.bcat), p(seq.out_wt), p(seq.out_b), p(emb_text), p(h0), p(mask_u8), p(text_len_i32), p(probs), p(picks),
        B, Lt, D, H, E, M, S, int(no_repeat), int(min_sentences), _lib.stream()), "mmb_decoder_greedy_constrained_fused")
    _count(1)
    return probs, picks


BEAM_MAX_WIDTH = 8


def decoder_beam_fwd(seq: DecoderSeq, emb_text, h0, mask_u8, text_len_i32, steps: int, width: int, no_repeat: bool = False,
                     min_sentences: int = 0, constrained: Optional[bool] = None):
    """The beam roll-out of ``steps`` decoder steps in eval mode with ``width`` slots per video as ONE launch (csrc/decoder_fused.cu;
    the rule is documented at mmb_decoder_beam_fused in include/mmbidaf_b200.h).  emb_text (B,Lt,E) fp32, h0 (B,H) fp32, mask_u8
    (B,M) uint8, text_len_i32 (B) int32 (the EOS row of video b is text_len[b] - 1).  Always the cluster kernel, whatever
    ``decoder_cut`` says: there is no chunk-cut beam.  ``no_repeat`` / ``min_sentences`` constrain the candidates (the rule at
    mmb_decoder_beam_constrained_fused); the constrained kernel runs when either is set, or when ``constrained`` says so.
    Returns (tokens (B,S,K) int64, parents (B,S,K) int32, scores (B,S,K) fp32, probs (B,S,K,M) fp32, best (B,S) int64,
    path (B,S) int32) -- ``best`` is slot 0's path after the last step, ``path`` its slot at every step."""
    lib = _lib.lib()
    B, Lt, D, H, E, M = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M
    dev = h0.device
    if not 1 <= int(width) <= BEAM_MAX_WIDTH:
        raise ValueError(f"decoder_beam_fwd: beam width {width} (1..{BEAM_MAX_WIDTH})")
    if int(steps) <= 0:
        raise ValueError(f"decoder_beam_fwd: {steps} steps")
    _check_constraints("decoder_beam_fwd", no_repeat, min_sentences)
    if emb_text.shape != (B, Lt, E) or h0.shape != (B, H) or mask_u8.shape != (B, M) or text_len_i32.shape != (B,):
        raise ValueError(f"decoder_beam_fwd: emb_text {tuple(emb_text.shape)}, h0 {tuple(h0.shape)}, mask {tuple(mask_u8.shape)}, "
                         f"text_len {tuple(text_len_i32.shape)} for B={B} Lt={Lt} E={E} H={H} M={M}")
    if text_len_i32.dtype != torch.int32:
        raise ValueError(f"decoder_beam_fwd: text_len {text_len_i32.dtype}, not int32")
    S, K = int(steps), int(width)
    tokens = torch.empty(B, S, K, device=dev, dtype=torch.int64)
    parents = torch.empty(B, S, K, device=dev, dtype=torch.int32)
    scores = torch.empty(B, S, K, device=dev, dtype=torch.float32)
    probs = torch.empty(B, S, K, M, device=dev, dtype=torch.float32)
    best = torch.empty(B, S, device=dev, dtype=torch.int64)
    path = torch.empty(B, S, device=dev, dtype=torch.int32)
    p = _lib.ptr
    args = (p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(seq.Wh4t), p(seq.bh4), p(seq.v1), p(seq.wc1), p(seq.v2),
            p(seq.wc2), p(seq.v1b), p(seq.v2b), p(seq.Wb13t), p(seq.vb1), p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(seq.Wcatt),
            p(seq.bcat), p(seq.out_wt), p(seq.out_b), p(emb_text), p(h0), p(mask_u8), p(text_len_i32), p(tokens), p(parents),
            p(scores), p(probs), p(best), p(path), B, Lt, D, H, E, M, K, S)
    if constrained is None:
        constrained = bool(no_repeat) or min_sentences > 0
    if constrained:
        _lib.check(lib.mmb_decoder_beam_constrained_fused(*args, int(no_repeat), int(min_sentences), _lib.stream()),
                   "mmb_decoder_beam_constrained_fused")
    else:
        _lib.check(lib.mmb_decoder_beam_fused(*args, _lib.stream()), "mmb_decoder_beam_fused")
    _count(1)
    return tokens, parents, scores, probs, best, path


SAMPLE_MAX_N, SAMPLE_MAX_TOP_K = 64, 8


def check_sampling(who: str, num_samples, temperature, top_k, top_p=1.0) -> None:
    """``num_samples`` an int in 1..64, ``temperature`` a finite number > 0, ``top_k`` an int in 0..8 (the rule at
    mmb_decoder_sample_fused in include/mmbidaf_b200.h), ``top_p`` a real in (0, 1] that stays above 0 in fp32 (the rule at
    mmb_decoder_sample_nucleus_fused)."""
    if isinstance(num_samples, bool) or not isinstance(num_samples, int) or not 1 <= num_samples <= SAMPLE_MAX_N:
        raise ValueError(f"{who}: num_samples {num_samples!r}, expected an int in 1..{SAMPLE_MAX_N}")
    if isinstance(temperature, bool) or not isinstance(temperature, (int, float)) or not math.isfinite(temperature) or temperature <= 0:
        raise ValueError(f"{who}: temperature {temperature!r}, expected a finite number > 0")
    if isinstance(top_k, bool) or not isinstance(top_k, int) or not 0 <= top_k <= SAMPLE_MAX_TOP_K:
        raise ValueError(f"{who}: top_k {top_k!r}, expected an int in 0..{SAMPLE_MAX_TOP_K}")
    if isinstance(top_p, bool) or not isinstance(top_p, (int, float)) or not 0 < top_p <= 1 or ctypes.c_float(top_p).value <= 0:
        raise ValueError(f"{who}: top_p {top_p!r}, expected a real in (0, 1]")


def decoder_sample_fwd(seq: DecoderSeq, emb_text, h0, mask_u8, text_len_i32, steps: int, num_samples: int, key: torch.Tensor,
                       temperature: float = 1.0, top_k: int = 0, no_repeat: bool = False, min_sentences: int = 0, top_p: float = 1.0):
    """N sampled roll-outs per video (the rule at mmb_decoder_sample_fused in include/mmbidaf_b200.h) as ONE launch of the cluster
    kernel, whatever ``decoder_cut`` says.  Inputs as :func:`decoder_greedy_constrained_fwd` (text_len_i32 may be None without a
    constraint), plus ``key`` (1) int64 on the device (:func:`rng_next_keys`, or a fill).  ``top_p`` < 1 draws from the nucleus
    (mmb_decoder_sample_nucleus_fused); 1 is the plain sampled launch.  Returns (probs (B,N,S,M), tokens (B,N,S) int64) -- each
    roll-out's distributions are the step kernel's, bit for bit."""
    lib = _lib.lib()
    B, Lt, D, H, E, M = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M
    dev = h0.device
    check_sampling("decoder_sample_fwd", num_samples, temperature, top_k, top_p)
    _check_constraints("decoder_sample_fwd", no_repeat, min_sentences)
    if int(steps) <= 0:
        raise ValueError(f"decoder_sample_fwd: {steps} steps")
    constrained = bool(no_repeat) or min_sentences > 0
    if emb_text.shape != (B, Lt, E) or h0.shape != (B, H) or mask_u8.shape != (B, M) or \
            (text_len_i32 is None and constrained) or (text_len_i32 is not None and text_len_i32.shape != (B,)):
        raise ValueError(f"decoder_sample_fwd: emb_text {tuple(emb_text.shape)}, h0 {tuple(h0.shape)}, mask {tuple(mask_u8.shape)}, "
                         f"text_len {None if text_len_i32 is None else tuple(text_len_i32.shape)} for B={B} Lt={Lt} E={E} H={H} M={M}")
    if text_len_i32 is not None and text_len_i32.dtype != torch.int32:
        raise ValueError(f"decoder_sample_fwd: text_len {text_len_i32.dtype}, not int32")
    if key.dtype != torch.int64 or key.numel() != 1 or key.device != dev:
        raise ValueError(f"decoder_sample_fwd: key {key.dtype} {tuple(key.shape)} on {key.device}, expected one int64 on {dev}")
    S, N = int(steps), int(num_samples)
    probs = torch.empty(B, N, S, M, device=dev, dtype=torch.float32)
    tokens = torch.empty(B, N, S, device=dev, dtype=torch.int64)
    p = _lib.ptr
    args = (p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(seq.Wh4t), p(seq.bh4), p(seq.v1), p(seq.wc1), p(seq.v2),
            p(seq.wc2), p(seq.v1b), p(seq.v2b), p(seq.Wb13t), p(seq.vb1), p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(seq.Wcatt),
            p(seq.bcat), p(seq.out_wt), p(seq.out_b), p(emb_text), p(h0), p(mask_u8), p(text_len_i32), p(key.contiguous()), p(probs),
            p(tokens), B, Lt, D, H, E, M, S, N, float(temperature), int(top_k), int(no_repeat), int(min_sentences))
    if top_p == 1.0:
        _lib.check(lib.mmb_decoder_sample_fused(*args, _lib.stream()), "mmb_decoder_sample_fused")
    else:
        _lib.check(lib.mmb_decoder_sample_nucleus_fused(*args, float(top_p), _lib.stream()), "mmb_decoder_sample_nucleus_fused")
    _count(1)
    return probs, tokens


def decoder_beam_sample_fwd(seq: DecoderSeq, emb_text, h0, mask_u8, text_len_i32, steps: int, width: int, key: torch.Tensor,
                            temperature: float = 1.0, no_repeat: bool = False, min_sentences: int = 0):
    """The stochastic beam roll-out (the rule at mmb_decoder_beam_sample_fused in include/mmbidaf_b200.h): ``width`` (1..8) distinct
    sequences per video, sampled without replacement, as ONE launch of the cluster kernel whatever ``decoder_cut`` says.  Inputs as
    :func:`decoder_beam_fwd`, plus ``key`` (1) int64 on the device (:func:`rng_next_keys` or :func:`seed_key`) and ``temperature``.
    Returns (tokens (B,S,K) int64, parents (B,S,K) int32, scores (B,S,K) fp32, probs (B,S,K,M) fp32, phi (B,S,K) fp32, keys (B,S,K)
    fp32, paths (B,K,S) int64, path_slots (B,K,S) int32, kappa (B) fp32) -- ``paths`` / ``path_slots`` are every final slot's tokens
    and slots (eos / -1 for an empty slot), ``kappa`` the threshold of the inclusion probabilities."""
    lib = _lib.lib()
    B, Lt, D, H, E, M = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M
    dev = h0.device
    if not 1 <= int(width) <= BEAM_MAX_WIDTH:
        raise ValueError(f"decoder_beam_sample_fwd: width {width} (1..{BEAM_MAX_WIDTH})")
    if int(steps) <= 0:
        raise ValueError(f"decoder_beam_sample_fwd: {steps} steps")
    if isinstance(temperature, bool) or not isinstance(temperature, (int, float)) or not math.isfinite(temperature) or temperature <= 0:
        raise ValueError(f"decoder_beam_sample_fwd: temperature {temperature!r}, expected a finite number > 0")
    _check_constraints("decoder_beam_sample_fwd", no_repeat, min_sentences)
    if emb_text.shape != (B, Lt, E) or h0.shape != (B, H) or mask_u8.shape != (B, M) or text_len_i32.shape != (B,):
        raise ValueError(f"decoder_beam_sample_fwd: emb_text {tuple(emb_text.shape)}, h0 {tuple(h0.shape)}, mask {tuple(mask_u8.shape)}, "
                         f"text_len {tuple(text_len_i32.shape)} for B={B} Lt={Lt} E={E} H={H} M={M}")
    if text_len_i32.dtype != torch.int32:
        raise ValueError(f"decoder_beam_sample_fwd: text_len {text_len_i32.dtype}, not int32")
    if key.dtype != torch.int64 or key.numel() != 1 or key.device != dev:
        raise ValueError(f"decoder_beam_sample_fwd: key {key.dtype} {tuple(key.shape)} on {key.device}, expected one int64 on {dev}")
    S, K = int(steps), int(width)
    tokens = torch.empty(B, S, K, device=dev, dtype=torch.int64)
    parents = torch.empty(B, S, K, device=dev, dtype=torch.int32)
    scores = torch.empty(B, S, K, device=dev, dtype=torch.float32)
    probs = torch.empty(B, S, K, M, device=dev, dtype=torch.float32)
    phi = torch.empty(B, S, K, device=dev, dtype=torch.float32)
    keys = torch.empty(B, S, K, device=dev, dtype=torch.float32)
    paths = torch.empty(B, K, S, device=dev, dtype=torch.int64)
    path_slots = torch.empty(B, K, S, device=dev, dtype=torch.int32)
    kappa = torch.empty(B, device=dev, dtype=torch.float32)
    p = _lib.ptr
    _lib.check(lib.mmb_decoder_beam_sample_fused(
        p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(seq.Wh4t), p(seq.bh4), p(seq.v1), p(seq.wc1), p(seq.v2),
        p(seq.wc2), p(seq.v1b), p(seq.v2b), p(seq.Wb13t), p(seq.vb1), p(seq.vb2), p(seq.vb1b), p(seq.vb2b), p(seq.Wcatt),
        p(seq.bcat), p(seq.out_wt), p(seq.out_b), p(emb_text), p(h0), p(mask_u8), p(text_len_i32), p(key.contiguous()), p(tokens),
        p(parents), p(scores), p(probs), p(phi), p(keys), p(paths), p(path_slots), p(kappa), B, Lt, D, H, E, M, K, S,
        float(temperature), int(no_repeat), int(min_sentences), _lib.stream()), "mmb_decoder_beam_sample_fused")
    _count(1)
    return tokens, parents, scores, probs, phi, keys, paths, path_slots, kappa


def sample_pick(probs: torch.Tensor, key: torch.Tensor, row_base: torch.Tensor, S: int, s: int, N: int = 1, temperature: float = 1.0,
                top_k: int = 0, eligible: Optional[torch.Tensor] = None, top_p: float = 1.0) -> torch.Tensor:
    """Steps 1 to 4 of the sampled pick (mmb_sample_pick) for the rows of ``probs`` (R, M) fp32: row r is sample r % N of video
    ``row_base[r]`` (R int32) at step ``s`` of ``S``; ``eligible`` (R, M) bool / uint8 limits the candidates; ``top_p`` < 1 draws
    from the nucleus (mmb_sample_pick_nucleus).  Returns picks (R) int64, -1 for a row without a candidate -- the roll-out kernel's
    pick, bit for bit."""
    check_sampling("sample_pick", N, temperature, top_k, top_p)
    if probs.dtype != torch.float32 or probs.dim() != 2 or not probs.is_cuda:
        raise ValueError(f"sample_pick: probs {probs.dtype} {tuple(probs.shape)} on {probs.device}, expected (R, M) fp32 on a GPU")
    R, M = probs.shape
    dev = probs.device
    if row_base.dtype != torch.int32 or row_base.numel() != R or row_base.device != dev:
        raise ValueError(f"sample_pick: row_base {row_base.dtype} {tuple(row_base.shape)} on {row_base.device} for {R} rows on {dev}")
    if key.dtype != torch.int64 or key.numel() != 1 or key.device != dev:
        raise ValueError(f"sample_pick: key {key.dtype} {tuple(key.shape)} on {key.device}, expected one int64 on {dev}")
    if eligible is not None and (eligible.shape != (R, M) or eligible.device != dev or
                                 eligible.dtype not in (torch.bool, torch.uint8)):
        raise ValueError(f"sample_pick: eligible {eligible.dtype} {tuple(eligible.shape)} on {eligible.device}, expected (R, M) = "
                         f"({R}, {M}) bool / uint8 on {dev}")
    if not 0 <= int(s) < int(S):
        raise ValueError(f"sample_pick: step {s} of {S}")
    picks = torch.empty(R, device=probs.device, dtype=torch.int64)
    args = (_lib.ptr(probs.contiguous()), _lib.ptr(_u8(eligible)), _lib.ptr(key.contiguous()), _lib.ptr(row_base.contiguous()), R, M,
            int(S), int(s), int(N), float(temperature), int(top_k), _lib.ptr(picks))
    if top_p == 1.0:
        _lib.check(_lib.lib().mmb_sample_pick(*args, _lib.stream()), "mmb_sample_pick")
    else:
        _lib.check(_lib.lib().mmb_sample_pick_nucleus(*args, float(top_p), _lib.stream()), "mmb_sample_pick_nucleus")
    _count(1)
    return picks


def seed_key(seed: int, device) -> torch.Tensor:
    """The sampling key of an int seed: splitmix64 of the seed (so that nearby seeds give unrelated streams), written by a device
    fill -- no host copy, so a CUDA graph captures it and every replay refills the same key."""
    z = (int(seed) + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    z ^= z >> 31
    return torch.full((1,), z - (1 << 64) if z >= 1 << 63 else z, dtype=torch.int64, device=device)


def greedy_select(argmax: torch.Tensor, text_len: torch.Tensor):
    """decode.greedy_search for a batch on the device: argmax (B,S) int64, text_len (B) int32 -> (sel (B,S) int32 = the chosen
    sentence indices padded with -1, count (B) int32)."""
    assert argmax.dtype == torch.int64 and text_len.dtype == torch.int32 and argmax.dim() == 2
    B, S = argmax.shape
    if text_len.numel() != B:
        raise ValueError(f"greedy_select: {text_len.numel()} lengths for {B} videos")
    sel = torch.empty(B, S, device=argmax.device, dtype=torch.int32)
    count = torch.empty(B, device=argmax.device, dtype=torch.int32)
    _lib.check(_lib.lib().mmb_greedy_select(_lib.ptr(argmax.contiguous()), _lib.ptr(text_len.contiguous()), _lib.ptr(sel),
                                            _lib.ptr(count), B, S, _lib.stream()), "mmb_greedy_select")
    _count(1)
    return sel, count


def decoder_step_bwd(seq: DecoderSeq, h, cell, coverage, probs, cell_out, saved, d_probs, d_h_out, d_cell_out,
                     d_att_cov, d_cov_out, d_proj_a, d_proj_i, vec_acc, scal_acc, target=None, d_lossvec=None,
                     att_cov=None, cov_out=None):
    """Backward of one decoder step.  ``d_proj_*`` (B,Lt,2H), ``vec_acc`` (B,6,2H), ``scal_acc`` (B,4) are accumulated
    in place.  Returns (d_h, d_cell, d_cov, d_logits, d_gates, d_ctx12, d_hw4, d_pre_b)."""
    lib = _lib.lib()
    B, Lt, D, H, E, M, nch = seq.B, seq.Lt, seq.D, seq.H, seq.E, seq.M, seq.nch
    hw, alpha, beta, ctx12, pb, xcat, gates = saved
    f32 = dict(device=h.device, dtype=torch.float32)
    p = _lib.ptr
    st = _lib.stream()
    c = lambda t: None if t is None else t.contiguous()
    d_logits_pad = torch.empty(B, seq.Mp, **f32)                               # zero-padded columns: aligned K below
    d_logits = d_logits_pad[:, :M]
    fused = target is not None and d_lossvec is not None
    g = c(d_lossvec) if fused else None                                        # (2, B): [d nll | d coverage term]
    gbuf = torch.empty(B, 4 * H + 4 * D, **f32)                                # [d_gates | d_hw4] side by side
    d_gates, d_hw4 = gbuf[:, :4 * H], gbuf[:, 4 * H:]
    d_cell = torch.empty(B, H, **f32)
    datt, d_pre_b, d_ctx12 = torch.empty(B, Lt, **f32), torch.empty(2, B, D, **f32), torch.empty(2, B, D, **f32)
    dcov_tot = torch.empty(B, Lt, **f32)
    cut = decoder_cut(B, Lt)
    if cut == "fused":
        # the WHOLE backward step as one cluster kernel (csrc/decoder_fused.cu): head, both text sweeps, d h.  "head" keeps the
        # round-2 cut (head kernel + chunk-parallel sweeps + library GEMM) as a cross-check.
        d_cov = torch.empty(B, Lt, **f32)
        d_h = torch.empty(B, H, **f32)
        _lib.check(lib.mmb_decoder_step_fused_bwd(
            p(probs), p(c(d_probs)), p(target if fused else None), p(g[0] if fused else None), p(g[1] if fused else None),
            p(seq.out_w), p(gates), p(cell), p(cell_out), p(c(d_h_out)), p(c(d_cell_out)), p(seq.Wcat_ctx), p(c(d_att_cov)),
            p(c(d_cov_out)), p(alpha), p(beta), p(ctx12), p(pb), p(hw), p(seq.vb1), p(seq.vb2), p(att_cov if fused else None),
            p(cov_out if fused else None), p(seq.Wb13), d_logits_pad.data_ptr(), seq.Mp, gbuf.data_ptr(), 4 * H + 4 * D, p(d_cell),
            p(datt), p(dcov_tot), p(d_pre_b), p(d_ctx12), p(vec_acc), p(scal_acc), p(seq.proj_a), p(seq.proj_i), p(seq.enc_a),
            p(seq.enc_i), p(coverage), p(seq.v1), p(seq.wc1), p(seq.v2), p(seq.wc2), p(d_proj_a), p(d_proj_i), p(d_cov),
            p(seq.Wh_stack), p(d_h), B, Lt, D, H, M, st), "mmb_decoder_step_fused_bwd")
        _count(1)
        return d_h, d_cell, d_cov, d_logits, d_gates, d_ctx12, d_hw4, d_pre_b
    if cut != "chunks":
        # everything up to the text sweeps as ONE cluster kernel (csrc/decoder_fused.cu: dec_bwd_head_kernel)
        _lib.check(lib.mmb_decoder_bwd_head(p(probs), p(c(d_probs)), p(target if fused else None), p(g[0] if fused else None),
                                            p(g[1] if fused else None), p(seq.out_w), p(gates), p(cell), p(cell_out), p(c(d_h_out)),
                                            p(c(d_cell_out)), p(seq.Wcat_ctx), p(c(d_att_cov)), p(c(d_cov_out)), p(alpha), p(beta),
                                            p(ctx12), p(pb), p(hw), p(seq.vb1), p(seq.vb2), p(att_cov if fused else None),
                                            p(cov_out if fused else None), p(seq.Wb13), d_logits_pad.data_ptr(), seq.Mp,
                                            gbuf.data_ptr(), 4 * H + 4 * D, p(d_cell), p(datt), p(dcov_tot), p(d_pre_b), p(d_ctx12),
                                            p(vec_acc), p(scal_acc), B, Lt, D, H, M, st), "mmb_decoder_bwd_head")
        _count(-2)                                                             # (one kernel where the chunk cut counts three)
    else:
        _lib.check(lib.mmb_decoder_out_softmax_bwd(p(probs), p(c(d_probs)), p(target if fused else None),
                                                   p(g[0] if fused else None), d_logits_pad.data_ptr(), seq.Mp, B, M, st),
                   "mmb_decoder_out_softmax_bwd")
        dh_logits = d_logits_pad @ seq.out_w_pad                               # (B, H)  library GEMM
        _lib.check(lib.mmb_decoder_cell_bwd(p(gates), p(cell), p(cell_out), p(dh_logits), p(c(d_h_out)), p(c(d_cell_out)),
                                            gbuf.data_ptr(), 4 * H + 4 * D, p(d_cell), B, H, st), "mmb_decoder_cell_bwd")
        d_xcat = d_gates @ seq.Wcat_ctx                                        # (B, D) = d ctx  library GEMM
        _lib.check(lib.mmb_decoder_attn_finish_bwd(p(d_xcat), D, p(c(d_att_cov)), p(c(d_cov_out)), p(alpha), p(beta),
                                                   p(ctx12), p(pb), p(hw), p(seq.vb1), p(seq.vb2), p(datt), p(d_pre_b),
                                                   p(d_ctx12), p(vec_acc), p(scal_acc), p(att_cov if fused else None),
                                                   p(cov_out if fused else None), p(g[1] if fused else None), p(dcov_tot),
                                                   B, Lt, D, st), "mmb_decoder_attn_finish_bwd")
        d_ctx12.baddbmm_(d_pre_b, seq.Wb13)                                    # += d_pre W_beta   library GEMM
    d_alpha, spart = torch.empty(B, 2, Lt, **f32), torch.empty(B, nch, 2, **f32)
    d_cov, colp = torch.empty(B, Lt, **f32), torch.empty(B, nch, 2, 3, D, **f32)
    separt = torch.empty(B, nch, 2, **f32)
    _lib.check(lib.mmb_decoder_attn_bwd(p(seq.proj_a), p(seq.proj_i), p(seq.enc_a), p(seq.enc_i), p(hw), p(coverage),
                                        p(alpha), p(beta), p(datt), p(d_ctx12), p(dcov_tot), p(d_pre_b), p(seq.v1),
                                        p(seq.wc1), p(seq.v2), p(seq.wc2), p(d_alpha), p(spart), p(d_proj_a), p(d_proj_i),
                                        p(d_cov), p(colp), p(separt), d_hw4.data_ptr(), 4 * H + 4 * D, p(vec_acc), p(scal_acc),
                                        p(seq.counters[1]), B, Lt, D, nch, st),
               "mmb_decoder_attn_bwd")
    d_h = gbuf @ seq.Wh_stack                                                  # (B, H)  library GEMM
    _count(5)
    return d_h, d_cell, d_cov, d_logits, d_gates, d_ctx12, d_hw4, d_pre_b


def masked_softmax_fwd(x2d: torch.Tensor, mask2d_u8: torch.Tensor, log_mode: bool) -> torch.Tensor:
    lib = _lib.lib()
    rows, n = x2d.shape
    y = torch.empty_like(x2d)
    _lib.check(lib.mmb_masked_softmax_fwd(_lib.ptr(x2d), _lib.ptr(mask2d_u8), _lib.ptr(y), rows, n, int(log_mode),
                                          _lib.stream()), "mmb_masked_softmax_fwd")
    _count(1)
    return y


def masked_softmax_bwd(y2d: torch.Tensor, dy2d: torch.Tensor, mask2d_u8: torch.Tensor, log_mode: bool) -> torch.Tensor:
    lib = _lib.lib()
    rows, n = y2d.shape
    dx = torch.empty_like(y2d)
    _lib.check(lib.mmb_masked_softmax_bwd(_lib.ptr(y2d), _lib.ptr(dy2d.contiguous()), _lib.ptr(mask2d_u8), _lib.ptr(dx),
                                          rows, n, int(log_mode), _lib.stream()), "mmb_masked_softmax_bwd")
    _count(1)
    return dx


def col_sum(a: torch.Tensor) -> torch.Tensor:
    """out (p) = a.sum(dim=0) for a tall (n, p) fp32 matrix: the bias gradients of the step (deterministic two-stage
    kernel, HBM-bound; ATen's dim-0 reduction runs at 0.4 - 1.3 TB/s on these shapes)."""
    n, p = a.shape
    if n == 0 or p == 0:
        raise RuntimeError(f"col_sum: empty matrix {tuple(a.shape)}")
    lib = _lib.lib()
    a = a.contiguous()
    R = lib.mmb_col_sum_blocks(n, p)
    partial = torch.empty(R, p, device=a.device, dtype=torch.float32)
    out = torch.empty(p, device=a.device, dtype=torch.float32)
    _lib.check(lib.mmb_col_sum(_lib.ptr(a), _lib.ptr(partial), _lib.ptr(out), n, p, _lib.stream()), "mmb_col_sum")
    _count(2)
    return out


def length_plan(lengths: torch.Tensor, L: int, M: int = 0, want_order: bool = False, out=None):
    """One launch from int32 device lengths (B): mask (B, L) bool, decoder mask (B, M) bool (if M), scheduling order (B) int32
    (if want_order) -- models.py:86-92, :119-123.  ``out`` = (mask, dec_mask, order) re-uses existing tensors (graph replay)."""
    lib = _lib.lib()
    assert lengths.dtype == torch.int32 and lengths.is_cuda
    B = lengths.numel()
    if out is None:
        mask = torch.empty(B, L, dtype=torch.bool, device=lengths.device)
        dec = torch.empty(B, M, dtype=torch.bool, device=lengths.device) if M else None
        order = torch.empty(B, dtype=torch.int32, device=lengths.device) if want_order else None
    else:
        mask, dec, order = out
    _lib.check(lib.mmb_length_plan(_lib.ptr(lengths), _lib.ptr(mask), _lib.ptr(dec), _lib.ptr(order), B, L, M if dec is not None else 0,
                                   _lib.stream()), "mmb_length_plan")
    _count(1)
    return mask, dec, order


def adadelta_clip_step(param: torch.Tensor, grad: torch.Tensor, square_avg: torch.Tensor, acc_delta: torch.Tensor,
                       grad_norm: torch.Tensor, max_norm: float, lr: float, rho: float, eps: float, weight_decay: float) -> None:
    """clip_grad_norm_(max_norm) + one Adadelta step (train.py:154-155, :110) in one pass over the flat buffers, in place."""
    lib = _lib.lib()
    _lib.check(lib.mmb_adadelta_clip_step(_lib.ptr(param), _lib.ptr(grad), _lib.ptr(square_avg), _lib.ptr(acc_delta),
                                          _lib.ptr(grad_norm), float(max_norm), float(lr), float(rho), float(eps),
                                          float(weight_decay), param.numel(), _lib.stream()), "mmb_adadelta_clip_step")
    _count(1)


def highway_fwd(pre: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """y = sigmoid(pre[:, :H]) * relu(pre[:, H:]) + (1 - sigmoid(pre[:, :H])) * x  (encoding.py:55-57)."""
    lib = _lib.lib()
    n, H = x.shape
    y = torch.empty_like(x)
    _lib.check(lib.mmb_highway_fwd(_lib.ptr(pre), _lib.ptr(x), _lib.ptr(y), n, H, _lib.stream()), "mmb_highway_fwd")
    _count(1)
    return y


def highway_bwd(pre: torch.Tensor, x: torch.Tensor, dy: torch.Tensor):
    lib = _lib.lib()
    n, H = x.shape
    d_pre, dx = torch.empty_like(pre), torch.empty_like(x)
    _lib.check(lib.mmb_highway_bwd(_lib.ptr(pre), _lib.ptr(x), _lib.ptr(dy.contiguous()), _lib.ptr(d_pre), _lib.ptr(dx),
                                   n, H, _lib.stream()), "mmb_highway_bwd")
    _count(1)
    return d_pre, dx
