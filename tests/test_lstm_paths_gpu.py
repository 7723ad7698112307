"""GPU: every instantiation the bi-LSTM launchers can run, against float64 (torch's packed LSTM, and the explicit loop of the oracle).

csrc/bilstm.cu, dispatch / pick_nb / launch:
  KS    8, 32 or 52 for H <= 16, <= 64, <= 104 (the register share of W_hh per lane)
  NB    1, or 2 when B * ndir > 148: two sequences share a CTA (the last CTA of an odd batch has an empty slot)
  KR    the backward keeps KR = 50 r values per half when KS == 52 and H <= 100, KR = KS otherwise
  DROP  the layer's output dropout applied inside both kernels (a key from ops.rng_next_keys)
  pair  MMB_LSTM_PAIR=1 runs the forward on a two-CTA cluster (bilstm_fwd_pair_kernel<KS>) when NB == 1, H >= 32 and the layer has no
        output dropout; every other forward takes the single-CTA kernel.  bilstm_fwd_pair_kernel<8> is compiled but never launched
        (H <= 16 < 32).  The trace kernels (MMB_LSTM_TRACE) are a debugging aid and not covered here.

Each case forces its kernels by construction; test_case_table_reaches_every_instantiation checks that with torch.profiler.

  case             B    L     in  H    ndir drop  pair order    lengths  forward               backward
  ks8-nb2          77   20    12  16   2    -     -    longest  ragged   <8,2,false,false>     <8,2,8,false>      odd B
  ks8-nb2-drop     80   20    12  9    2    0.3   -    longest  ragged   <8,2,false,true>      <8,2,8,true>
  ks32-nb2         77   24    20  33   2    -     -    none     pairs    <32,2,false,false>    <32,2,32,false>
  ks32-nb2-drop    90   24    20  64   2    0.2   -    longest  ragged   <32,2,false,true>     <32,2,32,true>
  kr50-nb2         80   40    64  100  2    -     -    none     pairs    <52,2,false,false>    <52,2,50,false>
  kr50-nb2-sorted  80   40    64  100  2    -     -    longest  pairs    <52,2,false,false>    <52,2,50,false>    other CTA pairs
  kr50-nb2-drop    77   40    64  100  2    0.2   -    none     pairs    <52,2,false,true>     <52,2,50,true>
  kr52-nb2         76   30    24  104  2    -     -    longest  ragged   <52,2,false,false>    <52,2,52,false>
  kr52-nb2-drop    79   30    24  101  2    0.35  -    none     pairs    <52,2,false,true>     <52,2,52,true>
  wave-149         149  16    16  100  2    0.2   -    longest  ragged   <52,2,false,true>     <52,2,50,true>     150 CTAs > 148 SMs
  config4-rank     128  1024  32  100  2    0.2   -    longest  ragged   <52,2,false,true>     <52,2,50,true>     config 4 per rank
  ks8-nb1          5    17    10  12   2    -     -    longest  ragged   <8,1,false,false>     <8,1,8,false>
  ks8-nb1-drop     6    17    10  16   2    0.2   -    longest  ragged   <8,1,false,true>      <8,1,8,true>
  ks32-nb1         7    25    20  48   2    -     -    none     ragged   <32,1,false,false>    <32,1,32,false>
  ks32-nb1-drop    7    25    20  40   2    0.5   -    longest  ragged   <32,1,false,true>     <32,1,32,true>
  kr50-nb1         9    30    40  100  2    -     -    longest  ragged   <52,1,false,false>    <52,1,50,false>
  kr50-nb1-drop    9    30    40  65   2    0.2   -    none     ragged   <52,1,false,true>     <52,1,50,true>
  kr52-nb1         4    20    16  102  2    -     -    longest  ragged   <52,1,false,false>    <52,1,52,false>
  kr52-nb1-drop    4    20    16  103  2    0.2   -    longest  ragged   <52,1,false,true>     <52,1,52,true>
  l1-nb2           80   1     16  100  2    0.2   -    longest  ragged   <52,2,false,true>     <52,2,50,true>     dW_hh = 0 branch
  l1-nb1           3    1     8   33   2    -     -    none     ragged   <32,1,false,false>    <32,1,32,false>
  zeros-nb2        78   15    12  40   2    0.2   -    longest  zeros    <32,2,false,true>     <32,2,32,true>     explicit loop
  zeros-nb1        6    9     12  100  2    -     -    none     zeros    <52,1,false,false>    <52,1,50,false>    explicit loop
  uni-nb1          6    20    12  100  1    -     -    longest  ragged   <52,1,false,false>    <52,1,50,false>
  uni-nb2          150  12    12  40   1    0.2   -    longest  ragged   <32,2,false,true>     <32,2,32,true>
  pair-h33         7    21    16  33   2    -     on   longest  ragged   pair<32>              <32,1,32,false>
  pair-h33-drop    7    21    16  33   2    0.2   on   longest  ragged   <32,1,false,true>     <32,1,32,true>
  pair-h100        5    30    24  100  2    -     on   none     ragged   pair<52>              <52,1,50,false>
  pair-h100-drop   5    30    24  100  2    0.2   on   longest  ragged   <52,1,false,true>     <52,1,50,true>

Lengths: ragged = uniform in 1..L with the first at L; pairs = by batch index, pairs (L, 1), (1, L), (m, m), (random, random) in turn, so
that with order none a length-1 sequence shares a CTA with a full-length one; zeros = ragged in 0..L with zero-length sequences, alone
and beside a full-length one in a CTA.  The float64 reference is torch's packed LSTM, except for the zero-length rows (it refuses length
0) and config4-rank (its CPU backward takes a minute there): those take an explicit loop of the oracle's cell, checked against both.
"""
import re
from collections import namedtuple

import pytest
import torch
from torch.nn.utils.rnn import PackedSequence, pack_padded_sequence, pad_packed_sequence

from conftest import grad_err, rel_err
from oracle import mmbidaf_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5           # forward, up to L = 300 as in test_lstm_gpu.py
LONG_TOL = 1e-4      # L >= 1000 (as test_long_lecture_gpu.py's 900-step recurrences)
GRAD_TOL = 5e-5
DROP_TOL = 1e-5      # dropped against un-dropped fed d y * mask / keep_prob
SMS = 148            # pick_nb: one wave of CTAs


def _fwd(ks, nb, drop):
    return f"bilstm_fwd_kernel<{ks},{nb},false,{'true' if drop else 'false'}>"


def _bwd(ks, nb, kr, drop):
    return f"bilstm_bwd_kernel<{ks},{nb},{kr},{'true' if drop else 'false'}>"


def _pair(ks):
    return f"bilstm_fwd_pair_kernel<{ks}>"


# every non-trace instantiation that dispatch() can launch, with and without MMB_LSTM_PAIR=1
REACHABLE = ({_fwd(ks, nb, d) for ks in (8, 32, 52) for nb in (1, 2) for d in (False, True)}
             | {_bwd(ks, nb, kr, d) for ks, kr in ((8, 8), (32, 32), (52, 50), (52, 52)) for nb in (1, 2) for d in (False, True)}
             | {_pair(32), _pair(52)})

Case = namedtuple("Case", "B L fan_in H ndir drop pair order rule kernels")
CASES = {
    "ks8-nb2": Case(77, 20, 12, 16, 2, 0.0, False, "longest", "ragged", {_fwd(8, 2, 0), _bwd(8, 2, 8, 0)}),
    "ks8-nb2-drop": Case(80, 20, 12, 9, 2, 0.3, False, "longest", "ragged", {_fwd(8, 2, 1), _bwd(8, 2, 8, 1)}),
    "ks32-nb2": Case(77, 24, 20, 33, 2, 0.0, False, None, "pairs", {_fwd(32, 2, 0), _bwd(32, 2, 32, 0)}),
    "ks32-nb2-drop": Case(90, 24, 20, 64, 2, 0.2, False, "longest", "ragged", {_fwd(32, 2, 1), _bwd(32, 2, 32, 1)}),
    "kr50-nb2": Case(80, 40, 64, 100, 2, 0.0, False, None, "pairs", {_fwd(52, 2, 0), _bwd(52, 2, 50, 0)}),
    "kr50-nb2-sorted": Case(80, 40, 64, 100, 2, 0.0, False, "longest", "pairs", {_fwd(52, 2, 0), _bwd(52, 2, 50, 0)}),
    "kr50-nb2-drop": Case(77, 40, 64, 100, 2, 0.2, False, None, "pairs", {_fwd(52, 2, 1), _bwd(52, 2, 50, 1)}),
    "kr52-nb2": Case(76, 30, 24, 104, 2, 0.0, False, "longest", "ragged", {_fwd(52, 2, 0), _bwd(52, 2, 52, 0)}),
    "kr52-nb2-drop": Case(79, 30, 24, 101, 2, 0.35, False, None, "pairs", {_fwd(52, 2, 1), _bwd(52, 2, 52, 1)}),
    "wave-149": Case(149, 16, 16, 100, 2, 0.2, False, "longest", "ragged", {_fwd(52, 2, 1), _bwd(52, 2, 50, 1)}),
    "config4-rank": Case(128, 1024, 32, 100, 2, 0.2, False, "longest", "ragged", {_fwd(52, 2, 1), _bwd(52, 2, 50, 1)}),
    "ks8-nb1": Case(5, 17, 10, 12, 2, 0.0, False, "longest", "ragged", {_fwd(8, 1, 0), _bwd(8, 1, 8, 0)}),
    "ks8-nb1-drop": Case(6, 17, 10, 16, 2, 0.2, False, "longest", "ragged", {_fwd(8, 1, 1), _bwd(8, 1, 8, 1)}),
    "ks32-nb1": Case(7, 25, 20, 48, 2, 0.0, False, None, "ragged", {_fwd(32, 1, 0), _bwd(32, 1, 32, 0)}),
    "ks32-nb1-drop": Case(7, 25, 20, 40, 2, 0.5, False, "longest", "ragged", {_fwd(32, 1, 1), _bwd(32, 1, 32, 1)}),
    "kr50-nb1": Case(9, 30, 40, 100, 2, 0.0, False, "longest", "ragged", {_fwd(52, 1, 0), _bwd(52, 1, 50, 0)}),
    "kr50-nb1-drop": Case(9, 30, 40, 65, 2, 0.2, False, None, "ragged", {_fwd(52, 1, 1), _bwd(52, 1, 50, 1)}),
    "kr52-nb1": Case(4, 20, 16, 102, 2, 0.0, False, "longest", "ragged", {_fwd(52, 1, 0), _bwd(52, 1, 52, 0)}),
    "kr52-nb1-drop": Case(4, 20, 16, 103, 2, 0.2, False, "longest", "ragged", {_fwd(52, 1, 1), _bwd(52, 1, 52, 1)}),
    "l1-nb2": Case(80, 1, 16, 100, 2, 0.2, False, "longest", "ragged", {_fwd(52, 2, 1), _bwd(52, 2, 50, 1)}),
    "l1-nb1": Case(3, 1, 8, 33, 2, 0.0, False, None, "ragged", {_fwd(32, 1, 0), _bwd(32, 1, 32, 0)}),
    "zeros-nb2": Case(78, 15, 12, 40, 2, 0.2, False, "longest", "zeros", {_fwd(32, 2, 1), _bwd(32, 2, 32, 1)}),
    "zeros-nb1": Case(6, 9, 12, 100, 2, 0.0, False, None, "zeros", {_fwd(52, 1, 0), _bwd(52, 1, 50, 0)}),
    "uni-nb1": Case(6, 20, 12, 100, 1, 0.0, False, "longest", "ragged", {_fwd(52, 1, 0), _bwd(52, 1, 50, 0)}),
    "uni-nb2": Case(150, 12, 12, 40, 1, 0.2, False, "longest", "ragged", {_fwd(32, 2, 1), _bwd(32, 2, 32, 1)}),
    "pair-h33": Case(7, 21, 16, 33, 2, 0.0, True, "longest", "ragged", {_pair(32), _bwd(32, 1, 32, 0)}),
    "pair-h33-drop": Case(7, 21, 16, 33, 2, 0.2, True, "longest", "ragged", {_fwd(32, 1, 1), _bwd(32, 1, 32, 1)}),
    "pair-h100": Case(5, 30, 24, 100, 2, 0.0, True, None, "ragged", {_pair(52), _bwd(52, 1, 50, 0)}),
    "pair-h100-drop": Case(5, 30, 24, 100, 2, 0.2, True, "longest", "ragged", {_fwd(52, 1, 1), _bwd(52, 1, 50, 1)}),
}


def _lengths(rule, B, L, gen):
    if rule == "pairs":
        lengths = []
        for c in range((B + 1) // 2):
            m, r = torch.randint(1, L + 1, (2,), generator=gen).tolist()
            lengths += [(L, 1), (1, L), (m, m), (m, r)][c % 4]
        return lengths[:B]
    lo = 0 if rule == "zeros" else 1
    lengths = torch.randint(lo, L + 1, (B,), generator=gen).tolist()
    lengths[0] = L
    if rule == "zeros":
        lengths[1] = 0                                   # beside the full-length sequence 0 in CTA 0 (order none)
        lengths[2:4] = [0, 0]                            # a CTA with no step at all
        lengths[5::7] = [0] * len(lengths[5::7])
    return lengths


Inputs = namedtuple("Inputs", "lengths x w g_out g_h g_c")


def _inputs(case):
    """Seeded CPU tensors: lengths, x (B, L, in), weights [w_ih, w_hh, b_ih, b_hh] * ndir (uniform in +-0.1, as test_lstm_gpu.py), and the
    incoming gradients of out (B, L, ndir H), h_n and c_n (B, ndir, H)."""
    c = CASES[case]
    gen = torch.Generator().manual_seed(sum(map(ord, case)) + 1000 * c.B + c.L)
    lengths = _lengths(c.rule, c.B, c.L, gen)
    w = [(torch.rand(*shape, generator=gen) - 0.5) * 0.2 for _ in range(c.ndir)
         for shape in ((4 * c.H, c.fan_in), (4 * c.H, c.H), (4 * c.H,), (4 * c.H,))]
    x = torch.randn(c.B, c.L, c.fan_in, generator=gen)
    g_out = torch.randn(c.B, c.L, c.ndir * c.H, generator=gen)
    g_h = torch.randn(c.B, c.ndir, c.H, generator=gen)
    g_c = torch.randn(c.B, c.ndir, c.H, generator=gen)
    return Inputs(lengths, x, w, g_out, g_h, g_c)


# ---- float64 references --------------------------------------------------------------------------------------------------------------

def _fp64_layer(x, lengths, w, ndir, loop=False):
    """One layer in float64 with autograd: (out (B, L, ndir H), h_n (B, ndir, H), c_n (B, ndir, H)), all in batch order.  torch's packed
    LSTM -- the library call of O.rnn_encoder_aten, here with one or two directions and c_n -- when every length is at least 1 and
    ``loop`` is off.  Else an explicit loop of the oracle's cell (O.lstm_cell) over the time steps, the whole batch per step, each
    sequence's state updated only at its own steps: a zero-length sequence gets zero outputs and zero states (the library refuses
    length 0), and the backward stays linear in L (the library's CPU backward at B = 128, L = 1024 takes a minute)."""
    B, L, _ = x.shape
    H = w[1].shape[1]
    if min(lengths) >= 1 and not loop:
        order = O.sort_order(lengths)
        packed = pack_padded_sequence(x[order], torch.Tensor(list(lengths))[order], batch_first=True)
        zeros = x.new_zeros(ndir, B, H)
        data, h_n, c_n = torch._VF.lstm(packed.data, packed.batch_sizes, (zeros, zeros), w, True, 1, 0.0, False, ndir == 2)
        out, _ = pad_packed_sequence(PackedSequence(data, packed.batch_sizes, None, None), batch_first=True, total_length=L)
        inverse = order.sort(0)[1]
        return out[inverse], h_n.transpose(0, 1)[inverse], c_n.transpose(0, 1)[inverse]
    n = torch.tensor(lengths).clamp(0, L).unsqueeze(1)
    outs, hs, cs = [], [], []
    for d in range(ndir):
        w_ih, w_hh, b_ih, b_hh = w[4 * d:4 * d + 4]
        xg = (x @ w_ih.t() + b_ih + b_hh).unbind(1)                    # (one tensor per step: no whole-input gradient per step)
        h = c = x.new_zeros(B, H)
        rows = [None] * L
        for t in (range(L - 1, -1, -1) if d else range(L)):
            live = t < n                                                # the reverse direction starts at each sequence's last step
            h1, c1 = O.lstm_cell(xg[t], h, c, w_hh)
            h, c = torch.where(live, h1, h), torch.where(live, c1, c)
            rows[t] = torch.where(live, h1, torch.zeros_like(h1))
        outs.append(torch.stack(rows, dim=1))
        hs.append(h)
        cs.append(c)
    return torch.cat(outs, dim=2), torch.stack(hs, dim=1), torch.stack(cs, dim=1)


def test_fp64_reference_is_the_oracle():
    """The float64 layer above against the oracle itself: O.rnn_encoder_aten (two directions; its h_n is left in sorted order, quirk Q3)
    and O.lstm_direction (the explicit loop, one direction and zero lengths)."""
    gen = torch.Generator().manual_seed(5)
    B, L, F, H = 6, 9, 5, 7
    x = torch.randn(B, L, F, generator=gen, dtype=torch.float64)
    w = [(torch.rand(*s, generator=gen, dtype=torch.float64) - 0.5) for _ in range(2) for s in ((4 * H, F), (4 * H, H), (4 * H,), (4 * H,))]
    lengths = [9, 3, 1, 9, 5, 3]
    p = {f"rnn.{k}_l0{sfx}": w[4 * d + i] for d, sfx in enumerate(("", "_reverse"))
         for i, k in enumerate(("weight_ih", "weight_hh", "bias_ih", "bias_hh"))}
    out, h_n, _ = _fp64_layer(x, lengths, w, 2)
    want_out, want_h = O.rnn_encoder_aten(p, x, lengths, 1)
    assert rel_err(out, want_out) < 1e-12 and rel_err(h_n[O.sort_order(lengths)], want_h) < 1e-12
    for lens, loop in ((lengths, False), (lengths, True), ([9, 0, 1, 0, 5, 3], False)):
        for ndir in (1, 2):
            out, h_n, c_n = _fp64_layer(x, lens, w[:4 * ndir], ndir, loop)
            for d in range(ndir):
                o, h = O.lstm_direction(x, lens, *w[4 * d:4 * d + 4], reverse=d == 1)
                assert rel_err(out[:, :, d * H:(d + 1) * H], o) < 1e-12 and rel_err(h_n[:, d], h) < 1e-12, (lens, loop, ndir, d)
            if 0 not in lens:                                           # c_n: the library call and the loop agree
                assert rel_err(c_n, _fp64_layer(x, lens, w[:4 * ndir], ndir, not loop)[2]) < 1e-12, (loop, ndir)


def _fp64(case, inp, mask, keep):
    """The case through _fp64_layer, dropout given the kernels' mask.  Returns out, y, h_n, c_n and two sets of gradients with respect
    to (x, *weights): of out.g + h_n.gh (what the autograd Function sees) and of out.g + h_n.gh + c_n.gc (the ops level, with d c_n)."""
    c = CASES[case]
    x64 = inp.x.double().requires_grad_(True)
    w64 = [t.double().requires_grad_(True) for t in inp.w]
    out, h_n, c_n = _fp64_layer(x64, inp.lengths, w64, c.ndir, loop=c.L >= 1000)
    y = out if mask is None else out * mask.cpu().double() / keep
    loss = (y * inp.g_out.double()).sum() + (h_n * inp.g_h.double()).sum()
    g_fn = torch.autograd.grad(loss, [x64, *w64], retain_graph=True)
    g_ops = torch.autograd.grad(loss + (c_n * inp.g_c.double()).sum(), [x64, *w64])
    return out.detach(), y.detach(), h_n.detach(), c_n.detach(), g_fn, g_ops


# ---- the kernels ---------------------------------------------------------------------------------------------------------------------

def _device(case, inp):
    """Device tensors of a case: lengths, order (longest first) or None, and the dropout key with its mask, or (None, None)."""
    from mmbidaf_b200 import ops
    c = CASES[case]
    len_d = torch.tensor(inp.lengths, dtype=torch.int32, device="cuda")
    ord_d = O.sort_order(inp.lengths).to(torch.int32).cuda() if c.order == "longest" else None
    if not c.drop:
        return len_d, ord_d, None, None
    ops.rng_seed(7000 + c.B + c.H)
    key = ops.rng_next_keys("cuda", 1)
    return len_d, ord_d, key, ops.dropout_mask(key, 1.0 - c.drop, (c.B, c.L, c.ndir * c.H))


def _fn_layer(case, inp, len_d, ord_d, key):
    """The autograd Function (functional.lstm_layer, as RNNEncoder calls it) forward and backward: (y, h_n, d x, [d weights])."""
    from mmbidaf_b200 import functional as Fn
    c = CASES[case]
    xin = inp.x.cuda().requires_grad_(True)
    w = [t.cuda().requires_grad_(True) for t in inp.w]
    y, h_n = Fn.lstm_layer(xin, len_d, ord_d, w, key, c.drop)
    ((y * inp.g_out.cuda()).sum() + (h_n * inp.g_h.cuda()).sum()).backward()
    torch.cuda.synchronize()
    return y.detach(), h_n.detach(), xin.grad, [t.grad for t in w]


def _inv_keep(keep):
    """1 / keep_prob as the kernels compute it: in float32."""
    return float(torch.tensor(1.0, dtype=torch.float32) / torch.tensor(keep, dtype=torch.float32))


_KERNEL = re.compile(r"(bilstm_(?:fwd_pair|fwd|bwd)_kernel<[^>]*>)")


def _launched(fn):
    """The bilstm kernels ``fn`` launches, as demangled names without spaces (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {re.sub(r"\s+", "", m.group(1)) for e in prof.events() for m in [_KERNEL.search(e.name)] if m}


def test_case_table_reaches_every_instantiation(monkeypatch):
    """Each case launches exactly the two kernels its row names, and the rows together launch every reachable instantiation."""
    assert len(REACHABLE) == 30
    seen = set()
    for case, c in CASES.items():
        assert (c.B * c.ndir > SMS) == any(",2," in k for k in c.kernels), case           # the row's NB follows pick_nb
        monkeypatch.setenv("MMB_LSTM_PAIR", "1" if c.pair else "0")
        inp = _inputs(case)
        len_d, ord_d, key, _ = _device(case, inp)
        got = _launched(lambda: _fn_layer(case, inp, len_d, ord_d, key))
        assert got == c.kernels, (case, got)
        seen |= got
    assert seen == REACHABLE, (sorted(REACHABLE - seen), sorted(seen - REACHABLE))


def _zero_past(t, lengths):
    """t (B, L, ...) is exactly zero past each length."""
    return all(bool((t[b, n:] == 0).all()) for b, n in enumerate(lengths))


@pytest.mark.parametrize("case", list(CASES))
def test_case_matches_fp64(case, monkeypatch):
    """Forward and backward of a case against float64, through the autograd Function and through ops.lstm_layer_fwd / _bwd:
      * out, y, h_n, c_n within 1e-5 (1e-4 at L >= 1000); out, y zero past each length, exactly;
      * d x and every weight and bias gradient within 5e-5 of fp64 autograd; at the ops level with a random d c_n as well (d x, d W_ih and
        d b computed in float64 from the kernel's d(pre-activation)), and d(pre-activation) zero past each length, exactly;
      * save = 0 (the eval forward) gives the save = 1 out, y, h_n and c_n bit for bit;
      * dropout: y == out * mask / keep_prob bit for bit (mask from ops.dropout_mask), out / h_n / c_n equal to the forward without
        dropout bit for bit, and d(pre-activation) within 1e-5 of the un-dropped backward fed d y * mask / keep_prob."""
    from mmbidaf_b200 import ops
    c = CASES[case]
    monkeypatch.setenv("MMB_LSTM_PAIR", "1" if c.pair else "0")
    tol = LONG_TOL if c.L >= 1000 else TOL
    gtol = LONG_TOL if c.L >= 1000 else GRAD_TOL
    inp = _inputs(case)
    B, L, H, nd, keep = c.B, c.L, c.H, c.ndir, 1.0 - c.drop
    len_d, ord_d, key, mask = _device(case, inp)
    want_out, want_y, want_h, want_c, g_fn, g_ops = _fp64(case, inp, mask, keep)
    zero_len = [b for b, n in enumerate(inp.lengths) if n == 0]

    # the autograd Function
    y, h_n, dx, dw = _fn_layer(case, inp, len_d, ord_d, key)
    errs = {"y": rel_err(y, want_y), "h_n": rel_err(h_n, want_h)}
    assert max(errs.values()) < tol, errs
    assert _zero_past(y, inp.lengths)
    gerrs = {"dx": grad_err(dx, g_fn[0])}
    gerrs.update({f"dw{i}": grad_err(g, want) for i, (g, want) in enumerate(zip(dw, g_fn[1:]))})
    assert max(gerrs.values()) < gtol, gerrs
    for b in zero_len:
        assert (h_n[b] == 0).all() and (dx[b] == 0).all(), b

    # the ops: forward with save = 1 and 0, backward with d c_n
    xd = inp.x.cuda()
    w_ih = torch.cat([inp.w[4 * d] for d in range(nd)]).cuda()
    w_hh = torch.stack([inp.w[4 * d + 1] for d in range(nd)]).cuda().contiguous()
    bias = torch.cat([inp.w[4 * d + 2] + inp.w[4 * d + 3] for d in range(nd)]).cuda()
    pre = torch.addmm(bias, xd.view(B * L, -1), w_ih.t()).view(B, L, nd, 4 * H)
    kp = keep if key is not None else 1.0
    gates = pre.clone()
    out, h_n, c_n, cell, y = ops.lstm_layer_fwd(gates, w_hh, len_d, ord_d, B, L, H, nd, True, key, kp)
    eval_out, eval_h, eval_c, eval_cell, eval_y = ops.lstm_layer_fwd(pre.clone(), w_hh, len_d, ord_d, B, L, H, nd, False, key, kp)
    torch.cuda.synchronize()
    errs = {"out": rel_err(out, want_out), "h_n": rel_err(h_n, want_h), "c_n": rel_err(c_n, want_c)}
    assert max(errs.values()) < tol, errs
    assert _zero_past(out, inp.lengths)
    assert eval_cell is None
    assert torch.equal(eval_out, out) and torch.equal(eval_h, h_n) and torch.equal(eval_c, c_n)
    g_out, g_h, g_c = inp.g_out.cuda(), inp.g_h.cuda(), inp.g_c.cuda()
    da = ops.lstm_layer_bwd(gates, cell, w_hh, len_d, ord_d, g_out, g_h, g_c, B, L, H, nd, key, kp)
    torch.cuda.synchronize()
    assert _zero_past(da, inp.lengths)
    da64 = da.double().cpu().view(B * L, nd * 4 * H)
    x64 = inp.x.double().view(B * L, -1)
    w_ih64 = w_ih.double().cpu()
    gerrs = {"dx": grad_err((da64 @ w_ih64).view(B, L, -1), g_ops[0])}
    for d in range(nd):
        rows = da64[:, d * 4 * H:(d + 1) * 4 * H]
        gerrs[f"dw_ih{d}"] = grad_err(rows.t() @ x64, g_ops[1 + 4 * d])
        gerrs[f"db{d}"] = grad_err(rows.sum(0), g_ops[3 + 4 * d])
    assert max(gerrs.values()) < gtol, gerrs
    if key is None:
        return

    # dropout, given the mask
    assert torch.equal(eval_y, y)
    assert torch.equal(y, torch.where(mask, out * _inv_keep(keep), torch.zeros_like(out)))
    assert _zero_past(y, inp.lengths)
    monkeypatch.setenv("MMB_LSTM_PAIR", "0")                             # the un-dropped twin on the single-CTA kernel too
    gates0 = pre.clone()
    out0, h0, c0, cell0, y0 = ops.lstm_layer_fwd(gates0, w_hh, len_d, ord_d, B, L, H, nd, True)
    assert y0 is None and torch.equal(out0, out) and torch.equal(h0, h_n) and torch.equal(c0, c_n)
    dy = torch.where(mask, g_out * _inv_keep(keep), torch.zeros_like(g_out))
    da0 = ops.lstm_layer_bwd(gates0, cell0, w_hh, len_d, ord_d, dy, g_h, g_c, B, L, H, nd)
    torch.cuda.synchronize()
    assert grad_err(da, da0) < DROP_TOL


# ---- bit-for-bit structure: a sequence's FMA chains do not depend on NB or on its CTA partner ---------------------------------------

def _ops_run(gates, w_hh, lengths, order, dout, dh, dc, H, key=None, keep=1.0):
    """Forward (save = 1) and backward of the ops on one batch: (out, y, h_n, c_n, d(pre-activation))."""
    from mmbidaf_b200 import ops
    B, L = gates.shape[:2]
    len_d = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    g = gates.clone()
    out, h_n, c_n, cell, y = ops.lstm_layer_fwd(g, w_hh, len_d, order, B, L, H, 2, True, key, keep)
    da = ops.lstm_layer_bwd(g, cell, w_hh, len_d, order, dout, dh, dc, B, L, H, 2, key, keep)
    torch.cuda.synchronize()
    return out, y, h_n, c_n, da


def _random_layer(B, L, H, seed):
    gen = torch.Generator().manual_seed(seed)
    lengths = _lengths("pairs", B, L, gen)
    t = [torch.randn(B, L, 2, 4 * H, generator=gen) * 0.6, (torch.rand(2, 4 * H, H, generator=gen) - 0.5) * 0.2,
         torch.randn(B, L, 2 * H, generator=gen), torch.randn(B, 2, H, generator=gen), torch.randn(B, 2, H, generator=gen)]
    return lengths, [v.cuda() for v in t]


@pytest.mark.parametrize("hid", [16, 40, 100, 104])
def test_two_sequences_per_cta_equal_one(hid, monkeypatch):
    """B = 80 (NB = 2, longest first) against the same sequences as sub-batches of 74 and 6 (NB = 1, no order): out, h_n, c_n and
    d(pre-activation) bit for bit.  Without dropout: the keep bits hash the batch position, which a sub-batch changes."""
    monkeypatch.setenv("MMB_LSTM_PAIR", "0")
    B, L = 80, 37
    lengths, (gates, w_hh, dout, dh, dc) = _random_layer(B, L, hid, 900 + hid)
    order = O.sort_order(lengths).to(torch.int32).cuda()
    full = _ops_run(gates, w_hh, lengths, order, dout, dh, dc, hid)
    parts = []
    for lo, hi in ((0, 74), (74, 80)):
        assert (hi - lo) * 2 <= SMS
        sub = [t[lo:hi].contiguous() for t in (gates, dout, dh, dc)]
        parts.append(_ops_run(sub[0], w_hh, lengths[lo:hi], None, sub[1], sub[2], sub[3], hid))
    for i, name in ((0, "out"), (2, "h_n"), (3, "c_n"), (4, "d pre-activation")):
        assert torch.equal(full[i], torch.cat([p[i] for p in parts])), name


@pytest.mark.parametrize("hid,drop", [(100, 0.2), (104, 0.0), (33, 0.2), (12, 0.3)])
def test_order_does_not_change_a_bit(hid, drop, monkeypatch):
    """B = 77 (NB = 2) with no order and with the longest-first order -- different CTA partners, the same batch positions, so dropout
    may stay on: out, y, h_n, c_n and d(pre-activation) bit for bit."""
    from mmbidaf_b200 import ops
    monkeypatch.setenv("MMB_LSTM_PAIR", "0")
    B, L = 77, 29
    lengths, (gates, w_hh, dout, dh, dc) = _random_layer(B, L, hid, 700 + hid)
    key = None
    if drop:
        ops.rng_seed(31 + hid)
        key = ops.rng_next_keys("cuda", 1)
    order = O.sort_order(lengths).to(torch.int32).cuda()
    a = _ops_run(gates, w_hh, lengths, None, dout, dh, dc, hid, key, 1.0 - drop)
    b = _ops_run(gates, w_hh, lengths, order, dout, dh, dc, hid, key, 1.0 - drop)
    for name, u, v in zip(("out", "y", "h_n", "c_n", "d pre-activation"), a, b):
        assert (u is None and v is None) or torch.equal(u, v), name


# ---- MMB_LSTM_PAIR=1 on a layer with output dropout --------------------------------------------------------------------------------

@pytest.mark.parametrize("hid", [33, 100])
def test_pair_switch_keeps_dropout(hid, monkeypatch):
    """With MMB_LSTM_PAIR=1 a layer with output dropout takes the single-CTA kernel (the pair kernel does not write y): y, out, h_n and
    c_n as with the switch off, bit for bit, through the ops and through the autograd Function.  The switched run goes first, onto
    freed NaN-filled blocks, so that a y the kernel leaves unwritten cannot hold an earlier run's values."""
    from mmbidaf_b200 import functional as Fn, ops
    B, L, F = 5, 30, 24
    gen = torch.Generator().manual_seed(hid)
    lengths = torch.randint(1, L + 1, (B,), generator=gen).tolist()
    lengths[0] = L
    w = [((torch.rand(*s, generator=gen) - 0.5) * 0.2).cuda() for _ in range(2) for s in ((4 * hid, F), (4 * hid, hid), (4 * hid,), (4 * hid,))]
    x = torch.randn(B, L, F, generator=gen).cuda()
    len_d = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    ord_d = O.sort_order(lengths).to(torch.int32).cuda()
    w_ih = torch.cat([w[0], w[4]])
    w_hh = torch.stack([w[1], w[5]]).contiguous()
    pre = torch.addmm(torch.cat([w[2] + w[3], w[6] + w[7]]), x.view(B * L, F), w_ih.t()).view(B, L, 2, 4 * hid)
    ops.rng_seed(4242 + hid)
    key = ops.rng_next_keys("cuda", 1)
    runs = {}
    for pair in ("1", "0"):
        monkeypatch.setenv("MMB_LSTM_PAIR", pair)
        junk = [torch.full((B, L, 2 * hid), float("nan"), device="cuda") for _ in range(6)]
        del junk
        out, h_n, c_n, _, y = ops.lstm_layer_fwd(pre.clone(), w_hh, len_d, ord_d, B, L, hid, 2, True, key, 0.8)
        junk = [torch.full((B, L, 2 * hid), float("nan"), device="cuda") for _ in range(6)]
        del junk
        fy, fh = Fn.lstm_layer(x, len_d, ord_d, [t.clone().requires_grad_(True) for t in w], key, 0.2)
        torch.cuda.synchronize()
        runs[pair] = (y, out, h_n, c_n, fy.detach(), fh.detach())
    for name, on, off in zip(("y", "out", "h_n", "c_n", "Function y", "Function h_n"), runs["1"], runs["0"]):
        assert torch.equal(on, off), name


# ---- a whole encoder ----------------------------------------------------------------------------------------------------------------

def test_whole_encoder_with_dropout_matches_fp64():
    """RNNEncoder(800, 100, 2, drop_prob=0.2) in training mode at B = 77 (NB = 2, image-encoder scale): the layer keys rebuilt from the
    seeded key stream, their masks from ops.dropout_mask; fp64 chains the layers with the masks between them.  Output, x_hidden (quirk
    Q3: rows in descending-length order), d x and every parameter gradient."""
    from mmbidaf_b200 import ops
    from mmbidaf_b200.layers import RNNEncoder
    B, L, F, H, p = 77, 130, 800, 100, 0.2
    torch.manual_seed(77)
    enc = RNNEncoder(F, H, 2, drop_prob=p).cuda().train()
    gen = torch.Generator().manual_seed(130)
    lengths = torch.randint(1, L + 1, (B,), generator=gen).tolist()
    lengths[0] = L
    x = torch.randn(B, L, F, generator=gen)
    g_out = torch.randn(B, L, 2 * H, generator=gen)
    g_h = torch.randn(B, 4, H, generator=gen)
    xin = x.cuda().requires_grad_(True)
    ops.rng_next_keys(xin.device, 1)                                     # the device's key state exists: rng_seed fills it
    ops.rng_seed(2024)
    keys = ops.rng_next_keys(xin.device, 2).clone()
    masks = [ops.dropout_mask(keys[k:k + 1], 1.0 - p, (B, L, 2 * H)).cpu().double() for k in range(2)]
    ops.rng_seed(2024)                                                   # the encoder draws the same two keys
    y, x_hidden = enc(xin, lengths)
    ((y * g_out.cuda()).sum() + (x_hidden * g_h.cuda()).sum()).backward()
    torch.cuda.synchronize()

    p64 = {n: t.detach().double().cpu().requires_grad_(True) for n, t in enc.named_parameters()}
    x64 = x.double().requires_grad_(True)
    cur, finals = x64, []
    for k in range(2):
        w = [p64[f"rnn.{kind}_l{k}{sfx}"] for sfx in ("", "_reverse") for kind in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
        out, h_n, _ = _fp64_layer(cur, lengths, w, 2)
        cur = out * masks[k] / (1.0 - p)
        finals.append(h_n)
    want_h = torch.cat(finals, dim=1)[O.sort_order(lengths)]
    ((cur * g_out.double()).sum() + (want_h * g_h.double()).sum()).backward()
    errs = {"out": rel_err(y, cur), "x_hidden": rel_err(x_hidden, want_h)}
    assert max(errs.values()) < TOL, errs
    assert _zero_past(y, lengths)
    gerrs = {"x": grad_err(xin.grad, x64.grad)}
    gerrs.update({n: grad_err(t.grad, p64[n].grad) for n, t in enc.named_parameters()})
    assert len(gerrs) == 17 and max(gerrs.values()) < GRAD_TOL, gerrs
