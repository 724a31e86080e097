"""ctypes binding of libfgnn_b200.so (C ABI declared in include/fgnn_b200.h).

The product path has no CPU fallback: if the shared library is missing or a tensor is not a
CUDA tensor, the call raises.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libfgnn_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "fgnn_b200.h")

FGNN_MAX_DEPTH = 8
FGNN_MAX_BLOCKS = 16
FP32, BF16, FP16 = 0, 1, 2
PRECISIONS = {"fp32": FP32, "bf16": BF16, "fp16": FP16}
FGNN_DETERMINISTIC = 0x100   # ORed into `precision` / passed as `flags`: fixed-order sums instead of atomics

c_float_p = C.POINTER(C.c_float)


class MlpParams(C.Structure):
    _fields_ = [("c_in", C.c_int32), ("c_out", C.c_int32), ("depth", C.c_int32),
                ("w", C.c_void_p * FGNN_MAX_DEPTH), ("b", C.c_void_p * FGNN_MAX_DEPTH),
                ("gn_w", C.c_void_p), ("gn_b", C.c_void_p), ("eps", C.c_float), ("constant_n", C.c_int32)]


class MlpGrads(C.Structure):
    _fields_ = [("w", C.c_void_p * FGNN_MAX_DEPTH), ("b", C.c_void_p * FGNN_MAX_DEPTH),
                ("gn_w", C.c_void_p), ("gn_b", C.c_void_p)]


class BlockParams(C.Structure):
    _fields_ = [("mlp1", MlpParams), ("mlp2", MlpParams), ("mlp3", MlpParams)]


class EmbedParams(C.Structure):
    _fields_ = [("num_blocks", C.c_int32), ("block", BlockParams * FGNN_MAX_BLOCKS)]


class BlockGrads(C.Structure):
    _fields_ = [("mlp1", MlpGrads), ("mlp2", MlpGrads), ("mlp3", MlpGrads)]


class EmbedGrads(C.Structure):
    _fields_ = [("num_blocks", C.c_int32), ("block", BlockGrads * FGNN_MAX_BLOCKS)]


class FgnnError(RuntimeError):
    pass


_lib = None
_lock = threading.Lock()

_vp, _i32, _sz = C.c_void_p, C.c_int32, C.c_size_t
_SIGNATURES = {
    "fgnn_version": (C.c_char_p, []),
    "fgnn_last_error": (C.c_char_p, []),
    "fgnn_device_supports_tcgen05": (C.c_int, []),
    "fgnn_launch_count": (C.c_int64, []),
    "fgnn_reset_launch_count": (None, []),
    "fgnn_mlp_workspace_bytes": (_sz, [_i32] * 5),
    "fgnn_mlp_fwd_f32": (C.c_int, [C.POINTER(MlpParams), _vp, _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_mlp_bwd_f32": (C.c_int, [C.POINTER(MlpParams), C.POINTER(MlpGrads), _vp, _vp, _vp, _vp, _i32, _i32,
                                   _vp, _vp, _sz, _vp]),
    "fgnn_mlp_workspace_bytes_ex": (_sz, [_i32] * 6),
    "fgnn_mlp_bwd_f32_ex": (C.c_int, [C.POINTER(MlpParams), C.POINTER(MlpGrads), _vp, _vp, _vp, _vp, _i32, _i32,
                                      _vp, _vp, _sz, _vp, _i32]),
    "fgnn_graphnorm_fwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_float, _i32, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_matmul_fwd_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_matmul_bwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_features_from_adjacency_u8": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp]),
    "fgnn_colmax_fwd_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_colmax_bwd_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_scores_fwd_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_scores_bwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fgnn_ce_workspace_bytes": (_sz, [_i32, _i32]),
    "fgnn_ce_argmax_fwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_ce_bwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "fgnn_lap_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "fgnn_scores_pair_fwd_f32": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "fgnn_scores_pair_bwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "fgnn_ce_pair_argmax_fwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "fgnn_ce_pair_bwd_f32": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "fgnn_lap_pair_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp]),
    "fgnn_generate_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "fgnn_generate_pairs_u8": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _i32, C.c_float, C.c_float, C.c_uint64, _vp, _sz, _vp]),
    "fgnn_head_workspace_bytes": (_sz, [_i32, _i32]),
    "fgnn_head_fwd": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_head_fwd_train": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_head_bwd": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_head_pair_workspace_bytes": (_sz, [_i32, _i32]),
    "fgnn_head_pair_fwd": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "fgnn_head_pair_fwd_train": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "fgnn_head_pair_bwd": (C.c_int, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "fgnn_embed_workspace_bytes": (_sz, [C.POINTER(EmbedParams), _i32, _i32, _i32]),
    "fgnn_embed_fwd": (C.c_int, [C.POINTER(EmbedParams), _i32, _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_embed_fwd_adjacency_u8": (C.c_int, [C.POINTER(EmbedParams), _i32, _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_embed_train_workspace_bytes": (_sz, [C.POINTER(EmbedParams), _i32, _i32, _i32]),
    "fgnn_embed_fwd_train": (C.c_int, [C.POINTER(EmbedParams), _i32, _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_embed_bwd": (C.c_int, [C.POINTER(EmbedParams), C.POINTER(EmbedGrads), _i32, _vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_adam_step_f32": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                     _i32, _vp, _vp, _vp]),
    "fgnn_profile_enable": (None, [C.c_int]),
    "fgnn_profile_reset": (None, []),
    "fgnn_profile_read": (C.c_int, [_i32, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "fgnn_debug_tc_matmul_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "fgnn_debug_tc_mlp_workspace_bytes": (_sz, [_i32] * 5),
    "fgnn_debug_tc_mlp": (C.c_int, [_i32, C.POINTER(MlpParams), _vp, _vp, _i32, _i32, _vp, _vp, _sz, _vp]),
    "fgnn_debug_tc_matmul": (C.c_int, [_i32, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _sz, _vp]),
}


def get_lib():
    """Load libfgnn_b200.so once.  Raises FgnnError (never falls back) if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise FgnnError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                                f"g.build()'` (or `make -C graph_neural_net_b200/csrc`). There is no CPU fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(status: int, what: str):
    if status != 0:
        msg = get_lib().fgnn_last_error().decode("utf-8", "replace")
        raise FgnnError(f"{what} failed (status {status}): {msg}")


def ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise FgnnError(f"{name}: fgnn_b200 operators run on CUDA tensors only (got a {t.device} tensor); "
                        "there is no CPU fallback")
    if t.dtype != torch.float32:
        raise FgnnError(f"{name}: expected float32, got {t.dtype}")
    return t.contiguous()


# ---- per-device scratch owned by torch's allocator ------------------------------------------
_workspaces = {}


def _scratch(nbytes: int, device) -> torch.Tensor:
    """torch.empty of nbytes uint8.  Under torch.use_deterministic_algorithms PyTorch fills new memory by default; the
    library never relies on its scratch's initial contents, so that fill (tens of GB for a training workspace) is
    skipped."""
    import torch.utils.deterministic as D
    fill = D.fill_uninitialized_memory
    D.fill_uninitialized_memory = False
    try:
        return torch.empty(int(nbytes), dtype=torch.uint8, device=device)
    finally:
        D.fill_uninitialized_memory = fill


def workspace(device, nbytes: int) -> torch.Tensor:
    """A reusable uint8 scratch tensor of at least nbytes on `device`, 1 KiB aligned (TMA / swizzled
    shared-memory tiles want 1024-byte aligned bases; torch only guarantees 512)."""
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = None
        _workspaces.pop(key, None)
        raw = _scratch(max(int(nbytes), 1 << 20) + 1024, device)
        off = (-raw.data_ptr()) % 1024
        buf = raw[off:off + raw.numel() - 1024]
        _workspaces[key] = buf
    return buf


def private_workspace(device, nbytes: int) -> torch.Tensor:
    """A 1 KiB-aligned uint8 tensor of nbytes that is NOT shared with other calls (the 16-bit training forward keeps
    its activations there until backward)."""
    raw = _scratch(int(nbytes) + 1024, device)
    off = (-raw.data_ptr()) % 1024
    return raw[off:off + int(nbytes)]


def release_workspaces():
    _workspaces.clear()
