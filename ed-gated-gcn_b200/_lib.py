"""ctypes binding of ``csrc/libedgcn.so`` (the C ABI declared in ``include/edgcn.h``).

There is no CPU or eager-PyTorch fallback: if the shared library is missing, or a
tensor is not on a CUDA device, the call raises.
"""
from __future__ import annotations

import ctypes
import threading
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# EDG_LIB = another build of the same ABI (A/B timing of kernel changes on one box); default: the in-tree library
LIB_PATH = os.environ.get("EDG_LIB") or os.path.join(_HERE, "csrc", "libedgcn.so")

F32, BF16 = 0, 1
ACT_NONE, ACT_SIGMOID, ACT_RELU = 0, 1, 2
PAD_MAX_PLUS_1, PAD_ZERO = 0, 1
DTYPES = {torch.float32: F32, torch.bfloat16: BF16}

_P, _I, _L, _Z, _F = c_void_p, c_int32, c_int64, c_size_t, c_float

# name -> (restype, argtypes); mirrors include/edgcn.h one to one
SIGNATURES = {
    "edg_version": (c_int, []),
    "edg_strerror": (c_char_p, [c_int]),
    "edg_last_cuda_error": (c_char_p, []),
    "edg_csr_from_heads": (c_int, [_P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "edg_csr_from_heads_edges_workspace": (_Z, [_I, _I, _I]),
    "edg_csr_from_heads_edges": (c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "edg_csr_from_dense_count": (c_int, [_P, c_int, _I, _I, _L, _L, _L, _P, _P, _P]),
    "edg_csr_from_dense_fill": (c_int, [_P, c_int, _I, _I, _L, _L, _L, _P, _P, _P]),
    "edg_tree_dist": (c_int, [_P, _P, _P, _P, _I, _I, _P, _P]),
    "edg_dist_pad": (c_int, [_P, _P, _I, _I, c_int, _P, _P]),
    "edg_aggregate": (c_int, [_P, c_int, _L, _P, c_int, _L, _I, _I, _P, _P, c_int, _P, _P, _I, _I, _P]),
    "edg_fused_tile_rows": (c_int, [_I, _I]),
    "edg_views_bwd_hmax": (c_int, [_P, _P, _P, _I, _I, _I, _P, _L, _P, c_int, _P]),
    "edg_head_du_workspace": (_Z, [_I]),
    "edg_head_du": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _P, _L, _P, _P, _P, _Z, _P]),
    "edg_tile_plan": (c_int, [_P, _P, _I, _I, _P, _P, _P]),
    "edg_gcn_layer": (c_int, [_P, _L, _I, _I, _P, _L, _I, _P, c_int, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P, _L, _P, _P,
                              _L, _P, c_int, _P, _Z, _P]),
    "edg_adam_multi": (c_int, [_I, _P, _P, _P, _P, _P, _P, c_float, c_float, c_float, c_float, c_float, c_float, _P]),
    "edg_block_head_fwd": (c_int, [_P, _L, _P, _L, _P, _L, _P, _L, _P, _L, _P, _P, _L, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "edg_block_head_bwd": (c_int, [_P, _P, _L, _P, _L, c_int, _P, _L, _P, _L, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _P,
                                   _P, _P]),
    "edg_block_head_wgrad_workspace": (_Z, [_I, _I, _I]),
    "edg_block_head_wgrad": (c_int, [_P, _P, _P, _L, _P, _L, _P, _L, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "edg_cross_entropy_workspace": (_Z, [_I]),
    "edg_cross_entropy_fwd": (c_int, [_P, _L, _P, _I, _I, _L, _P, _P, _P, _Z, _P]),
    "edg_cross_entropy_bwd": (c_int, [_P, _L, _P, _I, _I, _L, _P, _P, _P, _L, _P]),
    "edg_loss_combine": (c_int, [_P, _P, _P, c_float, c_float, c_float, _P, _P]),
    "edg_loss_combine_bwd": (c_int, [_P, c_float, c_float, c_float, _P, _P]),
    "edg_set_sm_budget": (c_int, [_I]),
    "edg_split_pitch": (_L, [_I]),
    "edg_split_f16": (c_int, [_P, _L, _I, _I, _P, _L, _P, _P]),
    "edg_linear_split_ok": (c_int, [_I, _I]),
    "edg_linear_split": (c_int, [_P, _L, _P, _I, _I, _P, _L, _P, _I, _P, c_int, _P, _L, _P]),
    "edg_wgrad_split_workspace": (_Z, [_I, _I, _I]),
    "edg_wgrad_split": (c_int, [_P, _L, _P, _I, _P, _L, _P, _I, _I, _P, _L, _P, c_int, _P, _Z, _P]),
    "edg_linear": (c_int, [_P, c_int, _L, _I, _I, _P, _L, _I, _P, c_int, _P, c_int, _L, _P]),
    "edg_wgrad_workspace": (_Z, [_I, _I, _I, c_int]),
    "edg_wgrad": (c_int, [_P, _L, _I, _P, _L, _I, c_int, _I, _P, _L, _P, c_int, c_int, _P, _Z, _P]),
    "edg_wgrad_batch_workspace": (_Z, [_I, _I, _I, _I]),
    "edg_wgrad_batch": (c_int, [_I, _P, _L, _I, _P, _L, _I, c_int, _I, _P, _L, _P, c_int, _P, _Z, _P]),
    "edg_mlp_chain": (c_int, [c_int, _I, _I, _P, _L, _P, _I, _I, _P]),
    "edg_cast_2d": (c_int, [_P, _L, _I, _I, _P, c_int, _L, c_int, _P]),
    "edg_cast_batch": (c_int, [_I, _P, _P, _P, _P, _P, _P, _P, c_int, _P]),
    "edg_trigger_gather": (c_int, [_P, c_int, _L, _P, _P, _I, _I, _P, _P, _L, c_int, _P]),
    "edg_trigger_scatter_add": (c_int, [_P, _P, _I, _I, _I, _P, _P, _P, c_int, _L, _P]),
    "edg_pool_fwd": (c_int, [_P, c_int, _L, _P, _I, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P]),
    "edg_diversity_fwd": (c_int, [_P, _I, _I, _I, _P, _P, _P]),
    "edg_views_bwd": (c_int, [_P, _P, _P, _P, c_int, _L, _I, _I, _I, _P, _P, _P, _L, _P, c_int, _P]),
    "edg_views_bwd_parts": (c_int, [_P, _P, _P, _P, c_int, _L, _I, _I, _I, _P, _P, _P, _L, _P, c_int, c_int, _P]),
    "edg_scores_kl_fwd": (c_int, [_P, c_int, _L, _P, _I, _I, _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "edg_head_bwd": (c_int, [_P, c_int, _L, _P, _I, _I, _P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, _L,
                             _P, _L, _P, _P, _P, _I, _P, _I, _P]),
    "edg_segment_mean": (c_int, [_P, c_int, _L, _P, _P, _I, _I, _P, c_int, _L, _P]),
    "edg_segment_mean_bwd": (c_int, [_P, c_int, _L, _P, _P, _I, _I, _P, _L, _I, _P]),
    "edg_lr_pool_fwd": (c_int, [_P, c_int, _L, _P, _P, _I, _I, _I, _P, _P, _P]),
    "edg_lr_pool_bwd": (c_int, [_P, _P, _I, _I, _P, c_int, _L, _P]),
    "edg_dropout_rows": (c_int, [_P, c_int, _L, _P, _L, _I, _I, _P, _I, _F, c_int, _P]),
    "edg_gate_rows": (c_int, [_P, c_int, _L, _P, _I, _I, _P, _P, c_int, _L, _P]),
    "edg_gate_rows_act": (c_int, [_P, c_int, _L, _P, _I, _I, _P, _P, c_int, _L, c_int, _P]),
    "edg_sigmoid_bwd": (c_int, [_P, c_int, _L, _P, c_int, _L, _I, _I, _P, c_int, _L, c_int, _P]),
    "edg_sum_scaled": (c_int, [_P, _L, _F, _P, _P]),
    "edg_colsum_workspace": (_Z, [_I, _I]),
    "edg_colsum": (c_int, [_P, c_int, _L, _I, _I, _P, c_int, _P, _Z, _P]),
    "edg_tree_dist_pairs": (c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _P, _P]),
    "edg_scores_kl_pairs_fwd": (c_int, [_P, c_int, _L, _P, _P, _P, _I, _I, _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P, _P,
                                        _P]),
    "edg_head_bwd_pairs": (c_int, [_P, c_int, _L, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, c_int, _P, _P, _P, _P, _P, _P,
                                   _P, _L, _P, _P, _P, _P, _P]),
    "edg_views_bwd_hmax_pairs": (c_int, [_P, _P, _P, _I, _I, _P, _I, _I, _P, _L, _P, c_int, _P]),
    "edg_trigger_scatter_add_pairs": (c_int, [_P, _P, _I, _I, _P, _I, _I, _P, _P, _P, c_int, _L, _P]),
    "edg_lr_pool_pairs_fwd": (c_int, [_P, c_int, _L, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "edg_lr_pool_pairs_bwd": (c_int, [_P, _P, _P, _P, _I, _I, _I, _P, c_int, _L, _P]),
    "edg_pool_drop_pairs": (c_int, [_P, c_int, _L, _P, _P, _P, _I, _I, _P, _I, _P, _I, _F, _P, _P, _P, _P]),
    "edg_scores_kl_drop_pairs_fwd": (c_int, [_P, c_int, _L, _P, _P, _P, _I, _I, _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P,
                                             _P, _P, _I, _F, _P]),
    "edg_head_bwd_drop_pairs": (c_int, [_P, c_int, _L, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, c_int, _P, _P, _P, _P,
                                        _P, _P, _P, _P, _L, _P, _P, _P, _P, _P, _I, _F, _P]),
    "edg_views_bwd_drop_pairs": (c_int, [_P, _P, _P, _P, _P, _I, _P, _P, _I, _P, _P, _I, _I, _P, _F, _P, c_int, _L, _P,
                                         c_int, _P]),
    "edg_scores_kl_sig_pairs_fwd": (c_int, [_P, c_int, _L, _P, _P, _P, _I, _I, _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P,
                                            _I, _F, _P]),
    "edg_head_bwd_sig_pairs": (c_int, [_P, c_int, _L, _P, _I, _P, _I, _P, _P, _P, _I, _I, _P, _P, _P, c_int, _P, _P, _P, _P,
                                       _P, _P, _P, _P, _L, _P, _P, _P, _P, _P, _I, _F, _P]),
}



class ChainStage(ctypes.Structure):
    """``edg_chain_stage`` of include/edgcn.h (one Linear of one gate chain)."""
    _fields_ = [("w", c_void_p), ("ldw", c_int64), ("bias", c_void_p), ("y", c_void_p), ("ldy", c_int64),
                ("out", c_void_p), ("ldo", c_int64), ("out_dtype", c_int)]


_lib = None


def load() -> ctypes.CDLL:
    """dlopen the in-tree shared library and attach the prototypes."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU or PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class EdgError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        lib = load()
        msg = lib.edg_strerror(rc).decode()
        if rc == -6:
            msg += ": " + lib.edg_last_cuda_error().decode()
        raise EdgError(f"libedgcn status {rc}: {msg}")


# kernels enqueued per C-ABI call (for the launch counter bench.py reports)
def _kernels_of(name: str, args) -> int:
    if name == "edg_wgrad":
        return 2 + (2 if args[11] else 0)
    if name == "edg_csr_from_heads":
        return 3
    if name == "edg_csr_from_heads_edges":
        return 0 if args[4] == 0 else (3 if (args[5] == 0 or args[6] == 0) else 7)
    if name == "edg_wgrad_split":
        return 4
    if name == "edg_block_head_wgrad":
        return 2
    if name == "edg_split_f16":
        return 2
    if name in ("edg_csr_from_dense_count", "edg_diversity_fwd", "edg_colsum", "edg_wgrad_batch", "edg_head_du"):
        return 2
    if name == "edg_gcn_layer":
        return 2 if args[23] else 1
    if name == "edg_adam_multi":
        return 2 if args[0] else 0
    if name == "edg_head_bwd_pairs":
        return 2 if args[22] else 1
    if name in ("edg_head_bwd_drop_pairs", "edg_head_bwd_sig_pairs"):
        return 2 if args[23] else 1
    if name == "edg_views_bwd_drop_pairs":
        return (1 if args[15] else 0) + (1 if args[18] else 0)
    if name == "edg_pool_drop_pairs":
        return (args[9] + 3) // 4
    if name == "edg_pool_fwd":
        return (args[7] + 3) // 4
    return 1


LAUNCHES = {"calls": 0, "kernels": 0}
HOOK = None          # bench.py installs a (name, args, fn) -> rc wrapper to time kernels with CUDA events


# Device of the call being assembled.  The argument list of `call(name, ptr(a), ptr(b), ..., stream())` is evaluated
# left to right before `call` runs: `ptr` records the device of the tensors it sees, `stream()` returns THAT device's
# current stream, and `call` launches with that device current.  The reference selects its GPU with `--device cuda:N`
# and never calls set_device (train.py:286), so tensors on cuda:1 with device 0 current is the normal case there.
_tls = threading.local()


def call(name: str, *args) -> None:
    fn = getattr(load(), name)
    LAUNCHES["calls"] += 1
    LAUNCHES["kernels"] += _kernels_of(name, args)
    dev = getattr(_tls, "dev", None)
    _tls.dev = None
    if dev is not None and dev != torch.cuda.current_device():
        with torch.cuda.device(dev):
            check(HOOK(name, args, fn) if HOOK is not None else fn(*args))
    else:
        check(HOOK(name, args, fn) if HOOK is not None else fn(*args))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise EdgError("libedgcn takes CUDA tensors only (there is no CPU path)")
    dev = getattr(_tls, "dev", None)
    if dev is None:
        _tls.dev = t.device.index
    elif dev != t.device.index:
        _tls.dev = None
        raise EdgError(f"tensors of one call live on different devices (cuda:{dev} and {t.device})")
    return t.data_ptr()


def stream():
    dev = getattr(_tls, "dev", None)
    return (torch.cuda.current_stream(dev) if dev is not None else torch.cuda.current_stream()).cuda_stream


def dt(t_or_dtype) -> int:
    d = t_or_dtype.dtype if isinstance(t_or_dtype, torch.Tensor) else t_or_dtype
    try:
        return DTYPES[d]
    except KeyError:
        raise EdgError(f"unsupported dtype {d}: the path computes in float32 or bfloat16") from None
