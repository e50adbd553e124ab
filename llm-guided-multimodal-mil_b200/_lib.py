"""ctypes binding of libmilb200.so (the C ABI declared in include/milb200.h).

There is NO CPU fallback: if the shared library is missing, or a tensor is not on a CUDA device, the
call raises.  PyTorch is used only for device memory, streams and autograd plumbing.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
# MILB200_LIB: developer hook for A/B runs of kernel variants (tools/build_variant.py); the product loads the in-tree build
LIB_PATH = os.environ.get("MILB200_LIB") or os.path.join(HERE, "libmilb200.so")

F32, BF16 = 0, 1
HOST_F32, HOST_BF16, HOST_F16, HOST_F64 = 0, 1, 2, 3
ACT_NONE, ACT_TANH, ACT_RELU, ACT_SIGMOID = 0, 1, 2, 3

_p, _i, _i64, _sz, _f = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float

# name -> (restype, argtypes); mirrors include/milb200.h one to one
SIGNATURES = {
    "milb200_version": (_i, []),
    "milb200_last_error": (C.c_char_p, []),
    "milb200_launch_count": (_i64, []),
    "milb200_count_launches": (None, [_i64]),
    "milb200_pack_gate_weights": (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _i, _p, _p]),
    "milb200_cast": (_i, [_p, _i, _p, _i, _i64, _p]),
    "milb200_transpose": (_i, [_p, _p, _i, _i, _i, _p]),
    "milb200_gated_score_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "milb200_gated_score_saves_activations": (_i, [_i, _i, _i]),
    "milb200_gated_score_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _p, _sz, _p]),
    "milb200_gated_score_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i64, _i, _i, _i,
                                     _p, _p, _p, _p, _p, _p, _sz, _p]),
    "milb200_gated_pool_bwd_supported": (_i, [_i, _i, _i]),
    "milb200_profile_enable": (None, [_i]),
    "milb200_debug_trace": (_i, [_p]),
    "milb200_profile_read": (_i, [_p, _i]),
    "milb200_pool_workspace_bytes": (_sz, [_i64, _i, _i]),
    "milb200_segment_softmax_pool_fwd": (_i, [_p, _p, _p, _i, _i64, _i, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "milb200_segment_softmax_pool_bwd": (_i, [_p, _p, _p, _i, _i64, _i, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "milb200_segment_softmax_pool_fwd_rowdot": (_i, [_p, _p, _p, _i, _i64, _i, _i, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "milb200_segment_softmax_pool_bwd_rowdot": (_i, [_p, _p, _i, _i64, _i, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "milb200_segment_sum_fwd": (_i, [_p, _p, _i, _i64, _i, _i, _p, _p, _p, _sz, _p]),
    "milb200_bag_broadcast": (_i, [_p, _p, _p, _i, _i64, _i, _i, _p, _p]),
    "milb200_dropout": (_i, [_p, _p, _i64, _f, C.c_uint64, C.c_uint64, _i, _p]),
    "milb200_linear_workspace_bytes": (_sz, [_i64, _i, _i, _i, _i]),
    "milb200_linear_fwd": (_i, [_p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _p, _sz, _p]),
    "milb200_linear_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _i, _p, _sz, _p]),
    "milb200_linear_f32out_fwd": (_i, [_p, _p, _p, _p, _i64, _i, _i, _i, _p]),
    "milb200_linear_f32out_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _p, _sz, _p]),
    "milb200_layernorm_workspace_bytes": (_sz, [_i64, _i]),
    "milb200_layernorm_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _p]),
    "milb200_layernorm_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _i, _p, _sz, _p]),
    "milb200_colsum": (_i, [_p, _i64, _i, _p, _i, _i, _p]),
    "milb200_attention_workspace_bytes": (_sz, [_i64, _i64, _i, _i, _i]),
    "milb200_attention_fwd": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i, _i, _i, _p, _sz, _p]),
    "milb200_attention_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i, _i, _i, _p, _sz, _p]),
    "milb200_clip_logits_fwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "milb200_clip_logits_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "milb200_cliploss_fwd_bwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "milb200_cosine_embedding_fwd_bwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "milb200_add": (_i, [_p, _p, _p, _i64, _i, _p]),
    "milb200_axpby": (_i, [_p, _p, _p, _i64, _f, _f, _i, _p]),
    "milb200_sinusoid_pe": (_i, [_p, _i64, _i, _i, _p]),
    "milb200_ct_tokens_fwd": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "milb200_ct_tokens_bwd": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "milb200_tape_arena_bytes": (_sz, [_p, _i, _p, _i, _i, _p]),
    "milb200_tape_workspace_bytes": (_sz, [_p, _i, _p, _i, _i, _i, _p]),
    "milb200_tape_forward": (_i, [_p, _i, _p, _i, _p, _i, _p, _p, _p, _p, _sz, _p, _sz, _i, _p, _p]),
    "milb200_tape_backward": (_i, [_p, _i, _p, _i, _p, _i, _p, _p, _p, _p, _p, _p, _p, _sz, _p, _sz, _i, _p, _p]),
    "milb200_adam_step": (_i, [_p, _p, _p, _p, _i64, _f, _f, _f, _f, _f, _f, _i, _p]),
    "milb200_sgd_step": (_i, [_p, _p, _i64, _f, _f, _f, _p]),
    "milb200_allreduce_update_symm": (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _p, _i64, _i, _f, _f, _f, _f, _f, _f, _i, _p, _p]),
    "milb200_adam_step_dev": (_i, [_p, _p, _p, _p, _i64, _f, _f, _f, _f, _f, _f, _p, _p]),
    "milb200_step_counter_inc": (_i, [_p, _p]),
    "milb200_pack_bags_offsets": (_i, [_p, _p, _i, _p, _p]),
    "milb200_pack_bags_host": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p, _i, _i64, _p, _i]),
    "milb200_sigmoid_bce_fwd_bwd": (_i, [_p, _p, _p, _p, _p, _i, _p]),
}



class TapeOp(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("kind", "in0", "in1", "in2", "out", "p0", "p1", "a0", "lane")]


class TapeSlot(C.Structure):
    _fields_ = [("rows", C.c_int64), ("cols", C.c_int32), ("external", C.c_int32)]


class TapeParam(C.Structure):
    _fields_ = [("offset", C.c_int64), ("rows", C.c_int32), ("cols", C.c_int32)]


class Segment(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("k_start", "len", "out_start", "tok_row")]


class Segments(C.Structure):
    _fields_ = [("seg", C.POINTER(Segment)), ("n_segs", C.c_int32), ("tokens", C.c_int32)]


def make_segments(rows, tokens):
    """rows: [(k_start, len, out_start, tok_row), ...] -> (Segments struct, keep-alive array).  Pass C.byref(struct)."""
    arr = (Segment * len(rows))(*[Segment(*map(int, r)) for r in rows])
    return Segments(arr, len(rows), int(tokens)), arr


OP_LINEAR, OP_ATTENTION, OP_LAYERNORM, OP_ADD = 1, 2, 3, 4
OP_JOIN, OP_HEADDIAG_U, OP_HEADDIAG_O, OP_T2I_POOL, OP_LN_SEG, OP_TOK_SCATTER = 5, 6, 7, 8, 9, 10
SLOT_EXTERNAL, SLOT_F32 = 1, 2
MAX_SEGMENTS = 16

_lib = None
_lock = threading.Lock()


class MilB200Error(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle.  Raises if the CUDA library has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise MilB200Error(
                        f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
                        "(nvcc, sm_100a). mil_b200 has no CPU or eager-PyTorch fallback.")
                h = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    if not hasattr(h, name):
                        continue  # entry points are added layer by layer; callers fail loudly on use
                    fn = getattr(h, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = h
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().milb200_last_error()
        raise MilB200Error(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise MilB200Error(f"unsupported dtype {t.dtype}: mil_b200 kernels take float32 or bfloat16")


def ptr(t):
    """Raw device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise MilB200Error("mil_b200 kernels need CUDA tensors (no CPU fallback exists)")
    if not t.is_contiguous():
        raise MilB200Error("mil_b200 kernels need contiguous tensors")
    return C.c_void_p(t.data_ptr())


_raw_stream_fn = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_get_device_fn = getattr(torch._C, "_cuda_getDevice", None)


def raw_stream() -> int:
    """cudaStream_t of PyTorch's current stream on the current device, as an int (the fast path avoids building a
    torch.cuda.Stream object per kernel call: that costs ~10 us of host time, a visible share of a launch-bound step)."""
    if _raw_stream_fn is not None and _get_device_fn is not None:
        return _raw_stream_fn(_get_device_fn())
    return torch.cuda.current_stream().cuda_stream


def stream_ptr():
    return C.c_void_p(raw_stream())


_ws = {}


def workspace(nbytes: int, device) -> torch.Tensor:
    """Grow-only scratch buffer per (device, stream); kernels of one stream run in order so a single
    buffer per stream is race-free."""
    key = (device.index if isinstance(device, torch.device) else torch.device(device).index, raw_stream())
    buf = _ws.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws[key] = buf
    return buf


def launch_count() -> int:
    return int(lib().milb200_launch_count())
