"""ctypes binding of libmmbidaf_b200.so (the C ABI declared in include/mmbidaf_b200.h).

There is no fallback: if the shared library is missing, or the device is not sm_100, every
op raises.  torch is used only for device memory and streams; all pointers handed to the
library are raw ``data_ptr()`` values of contiguous CUDA tensors.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmmbidaf_b200.so")

_lib: Optional[ctypes.CDLL] = None
_device_ok = False

c_void_p, c_int, c_float, c_size_t = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/mmbidaf_b200.h
SIGNATURES = {
    "mmb_version": [],
    "mmb_last_error": [],
    "mmb_device_supported": [],
    "mmb_bidaf_fwd": [c_void_p] * 10 + [c_float] + [c_void_p] * 6 + [c_int] * 5 + [c_void_p],
    "mmb_bidaf_workspace_bytes": [c_int] * 6,
    "mmb_bidaf_bwd": [c_void_p] * 11 + [c_float] + [c_void_p] * 13 + [c_int] * 5 + [c_void_p],
    "mmb_bidaf_bwd_workspace_bytes": [c_int] * 5,
    "mmb_bilstm_fwd": [c_void_p] * 8 + [c_int] * 5 + [c_void_p],
    "mmb_bilstm_bwd": [c_void_p] * 8 + [c_int] * 4 + [c_void_p],
    "mmb_bilstm_fwd_dropout": [c_void_p] * 10 + [c_float] + [c_int] * 5 + [c_void_p],
    "mmb_bilstm_bwd_dropout": [c_void_p] * 9 + [c_float] + [c_int] * 4 + [c_void_p],
    "mmb_dropout_mask": [c_void_p, c_float, ctypes.c_longlong, c_void_p, c_void_p],
    "mmb_rng_next": [c_void_p, c_void_p, c_int, c_void_p],
    "mmb_dropout_apply": [c_void_p, c_void_p, c_void_p, c_float, ctypes.c_longlong, c_void_p],
    "mmb_decoder_chunks": [c_int, c_int],
    "mmb_decoder_step_fused_fwd": [c_void_p] * 42 + [c_int] * 6 + [c_void_p],
    "mmb_decoder_greedy_fused": [c_void_p] * 28 + [c_int] * 8 + [c_void_p],
    "mmb_decoder_beam_fused": [c_void_p] * 31 + [c_int] * 8 + [c_void_p],
    "mmb_decoder_greedy_constrained_fused": [c_void_p] * 27 + [c_int] * 9 + [c_void_p],
    "mmb_decoder_beam_constrained_fused": [c_void_p] * 31 + [c_int] * 10 + [c_void_p],
    "mmb_decoder_beam_sample_fused": [c_void_p] * 35 + [c_int] * 8 + [c_float] + [c_int] * 2 + [c_void_p],
    "mmb_decoder_sample_fused":[c_void_p] * 28 + [c_int] * 8 + [c_float] + [c_int] * 3 + [c_void_p],
    "mmb_sample_pick": [c_void_p] * 4 + [c_int] * 5 + [c_float, c_int, c_void_p, c_void_p],
    "mmb_decoder_sample_nucleus_fused": [c_void_p] * 28 + [c_int] * 8 + [c_float] + [c_int] * 3 + [c_float, c_void_p],
    "mmb_sample_pick_nucleus": [c_void_p] * 4 + [c_int] * 5 + [c_float, c_int, c_void_p, c_float, c_void_p],
    "mmb_greedy_select": [c_void_p] * 4 + [c_int] * 2 + [c_void_p],
    "mmb_decoder_bwd_head": [c_void_p] * 25 + [c_int] + [c_void_p] + [c_int] + [c_void_p] * 7 + [c_int] * 5 + [c_void_p],
    "mmb_decoder_attn_fwd": [c_void_p] * 18 + [c_int] * 4 + [c_void_p],
    "mmb_decoder_attn_finish": [c_void_p] * 17 + [c_int] * 6 + [c_void_p],
    "mmb_decoder_cell_fwd": [c_void_p] * 4 + [c_int] * 2 + [c_void_p],
    "mmb_decoder_out_softmax": [c_void_p] * 5 + [c_int] * 2 + [c_void_p],
    "mmb_decoder_out_softmax_bwd": [c_void_p] * 5 + [c_int] * 3 + [c_void_p],
    "mmb_decoder_cell_bwd": [c_void_p] * 7 + [c_int] + [c_void_p] + [c_int] * 2 + [c_void_p],
    "mmb_decoder_attn_finish_bwd": [c_void_p, c_int] + [c_void_p] * 18 + [c_int] * 3 + [c_void_p],
    "mmb_decoder_step_fused_bwd": [c_void_p] * 25 + [c_int] + [c_void_p] + [c_int] + [c_void_p] * 21 + [c_int] * 5 + [c_void_p],
    "mmb_decoder_attn_bwd": [c_void_p] * 24 + [c_int] + [c_void_p] * 3 + [c_int] * 4 + [c_void_p],
    "mmb_highway_fwd": [c_void_p] * 3 + [ctypes.c_longlong, c_int, c_void_p],
    "mmb_highway_bwd": [c_void_p] * 5 + [ctypes.c_longlong, c_int, c_void_p],
    "mmb_length_plan": [c_void_p] * 4 + [c_int] * 3 + [c_void_p],
    "mmb_pack_segments": [c_void_p] * 3 + [c_int] + [c_void_p] * 2,
    "mmb_col_sum_blocks": [ctypes.c_longlong, c_int],
    "mmb_col_sum": [c_void_p] * 3 + [ctypes.c_longlong, c_int, c_void_p],
    "mmb_adadelta_clip_step": [c_void_p] * 5 + [c_float] * 5 + [ctypes.c_longlong, c_void_p],
    "mmb_masked_softmax_fwd": [c_void_p] * 3 + [ctypes.c_longlong, c_int, c_int, c_void_p],
    "mmb_masked_softmax_bwd": [c_void_p] * 4 + [ctypes.c_longlong, c_int, c_int, c_void_p],
}
_RESTYPES = {"mmb_last_error": ctypes.c_char_p, "mmb_bidaf_workspace_bytes": c_size_t,
             "mmb_bidaf_bwd_workspace_bytes": c_size_t}


DECODER_WEIGHT_FIELDS = ("W2", "b2", "Wc1", "bc1", "v1", "v1b", "W4", "b4", "Wc2", "bc2", "v2", "v2b",
                         "Wb1", "bb1", "Wb2", "bb2", "Wb3", "bb3", "Wb4", "bb4", "vb1", "vb1b", "vb2", "vb2b",
                         "lstm_w_ih", "lstm_w_hh", "lstm_b_ih", "lstm_b_hh", "out_w", "out_b")


def load() -> ctypes.CDLL:
    """Load the library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -m mmbidaf_b200.build` "
                               "(there is no CPU or PyTorch fallback for the mmbidaf_b200 kernels)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)            # AttributeError if the .so is stale
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, c_int)
        _lib = lib
    return _lib


def lib() -> ctypes.CDLL:
    """The library, after checking once that a B200 is the current device."""
    global _device_ok
    handle = load()
    if not _device_ok:
        if not torch.cuda.is_available():
            raise RuntimeError("mmbidaf_b200 needs a CUDA device (sm_100a); none is visible and there is no CPU path")
        if not handle.mmb_device_supported():
            raise RuntimeError(handle.mmb_last_error().decode())
        _device_ok = True
    return handle


def check(status: int, what: str) -> None:
    if status != 0:
        raise RuntimeError(f"{what} failed (status {status}): {load().mmb_last_error().decode()}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "mmbidaf_b200 ops take contiguous CUDA tensors"
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream
