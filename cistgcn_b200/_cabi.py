"""ctypes binding of the C-ABI declared in include/cistgcn_b200.h.

``lib()`` loads the nvcc-built ``cistgcn_b200/_lib/libcistgcn_b200.so`` (built by
``__graft_entry__.build()``) and raises if it is missing: the package has no fallback path.
``bind(path)`` only attaches the prototypes to an already-built library; the test-suite uses it for
the SIMT-emulator build of the same kernel sources (tests/emu), never the product.
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, Tuple

import torch

from .pack import DEFINES, ABI_VERSION

_LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib")
LIB_PATH = os.environ.get("CISTGCN_B200_LIB") or os.path.join(_LIB_DIR, "libcistgcn_b200.so")   # env: explicit path to another build of the same CUDA library
MAXB = DEFINES["CISTGCN_MAX_BLOCKS"]

_p = ctypes.c_void_p
_i32p = ctypes.POINTER(ctypes.c_int32)


class BlockTaps(ctypes.Structure):
    _fields_ = [("adj_s", _p), ("adj_t", _p), ("w1", _p), ("w2", _p)]


class Taps(ctypes.Structure):
    _fields_ = [("in_blocks", BlockTaps * MAXB), ("out_blocks", BlockTaps * MAXB),
                ("ctx_joints", _p), ("ctx_displacements", _p),
                ("ctx_seq_joints_n", _p), ("ctx_seq_joints_dims", _p)]


def _declared_exports():
    """Every function include/cistgcn_b200.h declares (the loader checks the library exports all of them)."""
    import re
    from .pack import _HEADER
    src = re.sub(r"/\*.*?\*/", "", open(_HEADER).read(), flags=re.S)
    return tuple(dict.fromkeys(re.findall(r"\b(cistgcn_\w+)\s*\(", src)))


EXPORTS = _declared_exports()
FLAG_FPN_FP32 = DEFINES["CISTGCN_FLAG_FPN_FP32"]
FLAG_DSTD_FUSED = DEFINES["CISTGCN_FLAG_DSTD_FUSED"]
FLAG_DSTD_TC = DEFINES["CISTGCN_FLAG_DSTD_TC"]
FLAG_DSTD_MIX_FFMA = DEFINES["CISTGCN_FLAG_DSTD_MIX_FFMA"]
FLAG_DSTD_ADJ_FFMA = DEFINES["CISTGCN_FLAG_DSTD_ADJ_FFMA"]
FLAG_DSTD_REDUCE_FFMA = DEFINES["CISTGCN_FLAG_DSTD_REDUCE_FFMA"]
PROFILE_KINDS = DEFINES["CISTGCN_PROFILE_KINDS"]


def bind(path: str) -> ctypes.CDLL:
    L = ctypes.CDLL(path)
    L.cistgcn_last_error.restype = ctypes.c_char_p
    L.cistgcn_last_error.argtypes = []
    L.cistgcn_abi_version.restype = ctypes.c_int
    L.cistgcn_abi_version.argtypes = []
    L.cistgcn_workspace_bytes.restype = ctypes.c_size_t
    L.cistgcn_workspace_bytes.argtypes = [_i32p, ctypes.c_int64]
    L.cistgcn_forward_f32.restype = ctypes.c_int
    L.cistgcn_forward_f32.argtypes = [_i32p, ctypes.c_int32, _p, _p, _p, _p, _p, _p, ctypes.c_size_t,
                                      ctypes.c_int64, ctypes.POINTER(Taps), _p]
    L.cistgcn_forward_bf16.restype = ctypes.c_int
    L.cistgcn_forward_bf16.argtypes = L.cistgcn_forward_f32.argtypes
    L.cistgcn_rollout_workspace_bytes.restype = ctypes.c_size_t
    L.cistgcn_rollout_workspace_bytes.argtypes = [_i32p, ctypes.c_int64]
    L.cistgcn_rollout_f32.restype = ctypes.c_int
    L.cistgcn_rollout_f32.argtypes = [_i32p, ctypes.c_int32, _p, _p, ctypes.c_int32, _p, _p, _p, _p, ctypes.c_size_t,
                                      ctypes.c_int64, _p]
    L.cistgcn_rollout_bf16.restype = ctypes.c_int
    L.cistgcn_rollout_bf16.argtypes = L.cistgcn_rollout_f32.argtypes
    L.cistgcn_dstd_block_f32.restype = ctypes.c_int
    L.cistgcn_dstd_block_f32.argtypes = [_i32p, _p, _p, _p, ctypes.c_int64, ctypes.POINTER(BlockTaps), _p, ctypes.c_size_t,
                                         ctypes.c_uint32, _p]
    L.cistgcn_dstd_block_workspace_bytes.restype = ctypes.c_size_t
    L.cistgcn_dstd_block_workspace_bytes.argtypes = [_i32p, ctypes.c_int64]
    L.cistgcn_fpn_chain_f32.restype = ctypes.c_int
    L.cistgcn_fpn_chain_f32.argtypes = [_i32p, ctypes.c_int32, _i32p, _p, _p, _p, ctypes.c_int64, ctypes.c_uint32, _p]
    L.cistgcn_profile_kind_name.restype = ctypes.c_char_p
    L.cistgcn_profile_kind_name.argtypes = [ctypes.c_int]
    L.cistgcn_tail_f32.restype = ctypes.c_int
    L.cistgcn_tail_f32.argtypes = [_i32p, _p, _p, _p, _p, _p, _p, _p, ctypes.c_int64, ctypes.POINTER(Taps), _p]
    L.cistgcn_mpjpe_f32.restype = ctypes.c_int
    L.cistgcn_mpjpe_f32.argtypes = [_p, _p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, _p, _p, _p]
    L.cistgcn_eval_metrics_f32.restype = ctypes.c_int
    L.cistgcn_eval_metrics_f32.argtypes = [_p, _p, _p, _p, ctypes.c_int32, _p, _p, _p, _p, ctypes.c_int64, ctypes.c_int32,
                                           ctypes.c_int32, ctypes.c_int32, _p]
    L.cistgcn_mpjpe_grouped_f32.restype = ctypes.c_int
    L.cistgcn_mpjpe_grouped_f32.argtypes = [_p, _p, _p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, _p, _p,
                                            _p]
    L.cistgcn_eval_metrics_grouped_f32.restype = ctypes.c_int
    L.cistgcn_eval_metrics_grouped_f32.argtypes = [_p, _p, _p, ctypes.c_int32, _p, _p, ctypes.c_int32, _p, _p, _p, _p, _p,
                                                   ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _p]
    L.cistgcn_augment_windows_f32.restype = ctypes.c_int
    L.cistgcn_augment_windows_f32.argtypes = [_p, _p, _p, _p, _p, _p, _p, _p, _p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                              ctypes.c_int32, _p]
    L.cistgcn_profile_enable.restype = ctypes.c_int
    L.cistgcn_profile_enable.argtypes = [ctypes.c_int]
    L.cistgcn_profile_read.restype = ctypes.c_int
    L.cistgcn_profile_read.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)]
    L.cistgcn_debug_phase_clocks.restype = ctypes.c_int
    L.cistgcn_debug_phase_clocks.argtypes = [_p]
    L.cistgcn_debug_stamp_iteration.restype = ctypes.c_int
    L.cistgcn_debug_stamp_iteration.argtypes = [ctypes.c_int]
    if L.cistgcn_abi_version() != ABI_VERSION:
        raise RuntimeError(f"cistgcn_b200: {path} has ABI {L.cistgcn_abi_version()}, header says {ABI_VERSION}; "
                           "rebuild with `python -c 'import __graft_entry__ as g; g.build()'`")
    return L


def _declared_train_exports():
    import re
    hdr = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "cistgcn_b200_train.h")
    src = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)
    return tuple(dict.fromkeys(re.findall(r"\b(cistgcn_\w+)\s*\(", src)))


TRAIN_EXPORTS = _declared_train_exports()


def bind_train(L: ctypes.CDLL) -> ctypes.CDLL:
    """Prototypes of include/cistgcn_b200_train.h (the differentiable path); idempotent."""
    if getattr(L, "_cistgcn_train_bound", False):
        return L
    i32, i64, f32, u64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_uint64
    protos = {
        "cistgcn_conv2d_fwd": [_p, _p, _p, _p, _p, _p],
        "cistgcn_conv2d_bwd_input": [_p, _p, _p, _p, _p],
        "cistgcn_conv2d_bwd_weight": [_p, _p, _p, _p, _p, _p, _p],
        "cistgcn_bn_fwd": [_p, _p, _p, _p, _p, _p, _p, _p, _p, i64, i32, i32, i32, f32, f32, _p],
        "cistgcn_bn_bwd": [_p, _p, _p, _p, _p, _p, _p, _p, _p, i64, i32, i32, i32, _p],
        "cistgcn_prelu_fwd": [_p, _p, _p, i64, i32, i32, i32, _p],
        "cistgcn_prelu_bwd": [_p, _p, _p, _p, _p, _p, i64, i32, i32, i32, _p],
        "cistgcn_act_fwd": [_p, _p, i64, i32, _p],
        "cistgcn_act_bwd": [_p, _p, _p, i64, i32, _p],
        "cistgcn_dropout": [_p, _p, i64, f32, u64, _p, _p],
        "cistgcn_counter_bump": [_p, _p],
        "cistgcn_copy4d": [_p, ctypes.POINTER(i64), _p, ctypes.POINTER(i64), ctypes.POINTER(i64), i32, _p],
        "cistgcn_axpby": [f32, _p, f32, _p, i64, _p],
        "cistgcn_gcn_fwd": [_p, _p, _p, i64, i32, i32, i32, i32, i32, _p],
        "cistgcn_gcn_bwd": [_p, _p, _p, _p, _p, i64, i32, i32, i32, i32, i32, _p],
        "cistgcn_outer_fwd": [_p, _p, _p, i64, i32, i32, i32, _p],
        "cistgcn_outer_bwd": [_p, _p, _p, _p, _p, i64, i32, i32, i32, _p],
        "cistgcn_stats_fwd": [_p, _p, i64, i32, i32, i32, _p],
        "cistgcn_stats_bwd": [_p, _p, _p, _p, i64, i32, i32, i32, _p],
        "cistgcn_spatial_mean_fwd": [_p, _p, i64, i32, i32, _p],
        "cistgcn_spatial_mean_bwd": [_p, _p, i64, i32, i32, i32, _p],
        "cistgcn_scale_fwd": [_p, _p, _p, i64, i32, i32, _p],
        "cistgcn_scale_bwd": [_p, _p, _p, _p, _p, i64, i32, i32, _p],
        "cistgcn_rowmax_fwd": [_p, _p, _p, i64, i32, _p],
        "cistgcn_rowmax_bwd": [_p, _p, _p, i64, i32, _p],
        "cistgcn_cumsum": [_p, _p, i64, i32, i32, i32, _p],
        "cistgcn_features_fwd": [_p, _p, i64, i32, i32, _p],
        "cistgcn_features_bwd": [_p, _p, _p, i64, i32, i32, _p],
        "cistgcn_mpjpe_bwd": [_p, _p, _p, i64, f32, _p],
        "cistgcn_adam_step": [_p, _p, _p, _p, i64, f32, f32, f32, f32, f32, i32, f32, _p],
    }
    sizes = {"cistgcn_conv2d_bwd_weight_scratch_floats": [_p], "cistgcn_bn_scratch_floats": [i32]}
    assert set(protos) | set(sizes) == set(TRAIN_EXPORTS), sorted((set(protos) | set(sizes)) ^ set(TRAIN_EXPORTS))
    for name, args in protos.items():
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = args
    for name, args in sizes.items():
        fn = getattr(L, name)
        fn.restype = ctypes.c_size_t
        fn.argtypes = args
    L._cistgcn_train_bound = True
    return L


_LIB = None


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"cistgcn_b200: CUDA extension {LIB_PATH} not found. Build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
                "There is no CPU / eager fallback for this path.")
        _LIB = bind(LIB_PATH)
    return _LIB


def check(rc: int, what: str, L: ctypes.CDLL = None):
    if rc != 0:
        L = L or lib()
        msg = L.cistgcn_last_error()
        raise RuntimeError(f"cistgcn_b200: {what} failed ({rc}): {msg.decode() if msg else '?'}")


def make_taps(geom, B: int, device) -> Tuple[Taps, Dict[str, torch.Tensor]]:
    """Allocate the interpretability outputs named like the reference's module attributes."""
    t = Taps()
    out: Dict[str, torch.Tensor] = {}

    def new(name, *shape):
        out[name] = torch.empty(*shape, device=device, dtype=torch.float32)
        return out[name].data_ptr()

    T, V, To = geom.input_n, geom.joints, geom.output_n
    for i in range(len(geom.in_chain) - 1):
        p, co = f"st_gcnns.{i}", geom.in_chain[i + 1]
        bt = t.in_blocks[i]
        if geom.in_interp[i]:
            bt.adj_s = new(p + ".dsgn.Adj", B, V, T, T)
            bt.adj_t = new(p + ".tsgn.Adj", B, T, V, V)
        bt.w1 = new(p + ".w1", B, co)
        bt.w2 = new(p + ".w2", B, co)
    for i in range(len(geom.out_chain) - 1):
        p, co = f"st_gcnns_o.{i}", geom.out_chain[i + 1]
        bt = t.out_blocks[i]
        if geom.out_interp[i]:
            bt.adj_s = new(p + ".dsgn.Adj", B, To, V, V)      # block sees "T" = V, "V" = To
            bt.adj_t = new(p + ".tsgn.Adj", B, V, To, To)
        bt.w1 = new(p + ".w1", B, co)
        bt.w2 = new(p + ".w2", B, co)
    t.ctx_joints = new("context_layer.joints", B, V)
    t.ctx_displacements = new("context_layer.displacements", B, To)
    t.ctx_seq_joints_n = new("context_layer.seq_joints_n", B, To, V)
    t.ctx_seq_joints_dims = new("context_layer.seq_joints_dims", B, 3, To, V)
    return t, out
