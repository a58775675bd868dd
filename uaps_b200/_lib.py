"""ctypes binding of libuaps_b200.so (the C ABI declared in include/uaps_b200.h).

There is no fallback: if the shared library is missing or a call fails, this raises.
Pointers cross the boundary as plain integers (``tensor.data_ptr()``) and the stream as the raw
``cudaStream_t`` of torch's current stream, so the kernels run in stream order with torch's own
work and can be captured into CUDA graphs.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

from . import stepctx as _stepctx

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libuaps_b200.so")

KMAX, CMAX = 6, 8
LOSS_EXACT = 1
SC_LOSS_U, SC_PS_LOSS, SC_L_UNCERT, SC_CW1, SC_CW2, SC_INV_N, SC_MEAN_CE, SC_MEAN_DICE, SC_BASE = 0, 1, 2, 3, 4, 5, 6, 7, 8

_vp, _i, _i64, _u64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float, C.c_double
ABI_VERSION = 2
STEP_USLOTS = 16


class PackJobStruct(C.Structure):
    """Mirror of ``UapsPackJob`` (include/uaps_b200.h)."""
    _fields_ = [("w", C.c_void_p), ("w_packed", C.c_void_p), ("cout", C.c_int), ("cin1", C.c_int), ("cin2", C.c_int),
                ("ks", C.c_int), ("transpose", C.c_int), ("fold", C.c_int)]


class StepStateStruct(C.Structure):
    """Mirror of ``UapsStepState`` (include/uaps_b200.h): the device-resident per-iteration scalars."""
    _fields_ = [("iter", C.c_uint64), ("key_rank", C.c_uint64), ("key_shared", C.c_uint64), ("adam_step", C.c_uint64),
                ("xchg_base", C.c_uint32), ("xchg_next", C.c_uint32), ("skipped", C.c_uint32), ("n_skipped", C.c_uint32),
                ("lr", C.c_float), ("adam_step_size", C.c_float), ("adam_inv_bc2_sqrt", C.c_float), ("reserved", C.c_float),
                ("mix_w", C.c_float * 8), ("cw1", C.c_float), ("cw2", C.c_float), ("u", C.c_float * STEP_USLOTS)]

_SIGNATURES = {
    "uaps_abi_version": (_i, []),
    "uaps_error_string": (C.c_char_p, [_i]),
    "uaps_loss_sums_count": (_i, [_i, _i]),
    "uaps_loss_scalars_count": (_i, [_i, _i]),
    "uaps_loss_workspace_bytes": (C.c_size_t, [_i, _i]),
    "uaps_loss_pass1": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "uaps_step_begin": (_i, [_vp, _u64, _u64, _i, _i, _d, _d, _d, _i, _i, _f, _f, _vp]),
    "uaps_loss_pass1_scalars": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _f, _f, _vp, _vp, _vp]),
    "uaps_loss_pass1_exchange": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, C.c_uint, _i64,
                                      _f, _f, _vp, _vp, _vp, _vp]),
    "uaps_xchg_mailbox_bytes": (C.c_size_t, []),
    "uaps_xchg_alloc": (_i, [_vp]),
    "uaps_xchg_free": (_i, [_vp]),
    "uaps_xchg_export": (_i, [_vp, _vp]),
    "uaps_xchg_import": (_i, [_vp, _vp]),
    "uaps_xchg_close": (_i, [_vp]),
    "uaps_xchg_status": (_i, [_vp, _vp, _vp]),
    "uaps_loss_finalize": (_i, [_vp, _i, _i, _i64, _f, _f, _i, _vp, _vp]),
    "uaps_loss_pass2": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "uaps_ensemble_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i64]),
    "uaps_ensemble_head": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "uaps_feature_noise": (_i, [_vp, _vp, _u64, _f, _vp, _i, _i64, _vp]),
    "uaps_dropout": (_i, [_vp, _vp, _u64, _d, _vp, _i64, _vp]),
    "uaps_fdrop_stats": (_i, [_vp, _i, _i, _i64, _vp, _vp, _vp]),
    "uaps_fdrop_apply": (_i, [_vp, _vp, _vp, _f, _vp, _i, _i, _i64, _vp]),
    "uaps_perturb3": (_i, [_vp, _vp, _vp, _u64, _f, _d, _vp, _vp, _f, _vp, _vp, _vp, _i, _i, _i64, _vp]),
    "uaps_fdrop_stats_nhwc": (_i, [_vp, _i, _i, _i64, _vp, _vp, _vp]),
    "uaps_perturb3_nhwc": (_i, [_vp, _u64, _f, _d, _vp, _vp, _f, _vp, _vp, _vp, _i, _i, _i64, _vp, _vp, _vp]),
    "uaps_perturb3_nhwc_bwd": (_i, [_vp, _vp, _vp, _u64, _f, _d, _vp, _vp, _f, _vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "uaps_upsample2x_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "uaps_maxpool2_nhwc": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "uaps_nchw_f32_to_nhwc_bf16": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "uaps_nchw_f32_to_nhwc_bf16_sums_nrep": (_i, []),
    "uaps_nchw_f32_to_nhwc_bf16_sums": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "uaps_bn_stats_nhwc": (_i, [_vp, _i64, _i, _vp, _vp, _vp]),
    "uaps_bn_act_nhwc": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _d, _u64, _vp, _vp, _vp, _i64, _i, _vp, _i, _vp]),
    "uaps_conv_fprop_bn": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "uaps_bn_act_bwd_nhwc": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _f, _d, _u64, _vp, _vp, _vp, _vp, _vp, _i64, _i, _vp, _vp]),
    "uaps_conv_packed_bytes": (C.c_size_t, [_i, _i, _i, _i, _i]),
    "uaps_conv_pack_weights": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "uaps_conv_pack_job_bytes": (C.c_size_t, []),
    "uaps_conv_pack_plan": (_i, [_vp, _i, _vp, _vp]),
    "uaps_conv_pack_run": (_i, [_vp, _i, _i, _vp]),
    "uaps_conv_fprop": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "uaps_conv_fprop_act": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _f, _vp]),
    "uaps_conv_wgrad_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i, _i]),
    "uaps_conv_wgrad": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, C.c_size_t, _vp]),
    "uaps_adam_step": (_i, [_vp, _vp, _vp, _vp, _i64, _i64, _f, _f, _f, _f, _f, _vp, _vp, _vp]),
    "uaps_confusion": (_i, [_vp, _vp, _i, _i, _i64, _vp, _vp]),
    "uaps_val_workspace_bytes": (C.c_size_t, [_i, _i, _i64]),
    "uaps_val_counts": (_i, [_vp, _vp, _i, _i, _i64, _vp, C.c_size_t, _vp]),
    "uaps_val_fold": (_i, [_vp, C.c_size_t, _i, _i, _i64, _vp, _i, _vp, _vp]),
    "uaps_peer_alloc": (_i, [_vp, C.c_size_t]),
    "uaps_peer_free": (_i, [_vp]),
    "uaps_grad_reduce_adam": (_i, [_vp, _vp, _vp, _vp, _i64, _vp, _i, _i, _i64, _f, _f, _f, _f, _f, _vp, _vp, _vp]),
    "uaps_perturb3_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _u64, _f, _d, _vp, _vp, _f, _vp, _i, _i, _i64, _vp]),
    "uaps_unet_params_count": (C.c_size_t, [_i, _i]),
    "uaps_unet_infer_state_bytes": (C.c_size_t, [_i, _i]),
    "uaps_unet_infer_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i]),
    "uaps_unet_infer_prepare": (_i, [_vp, _i, _i, _vp, C.c_size_t, _vp]),
    "uaps_unet_infer_run": (_i, [_vp, C.c_size_t, _i, _i, _vp, _i, _i, _i, _vp, C.c_size_t, _vp, _vp, _vp]),
    "uaps_unet_infer_layer": (_i, [_i, _i, _i, _vp, _vp, _vp, _vp]),
    "uaps_unet_ensemble_params_count": (C.c_size_t, [_i, _i, _i]),
    "uaps_unet_ensemble_state_bytes": (C.c_size_t, [_i, _i, _i]),
    "uaps_unet_ensemble_draws_count": (C.c_size_t, [_i]),
    "uaps_unet_ensemble_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i, _i, _i]),
    "uaps_unet_ensemble_prepare": (_i, [_vp, _i, _i, _i, _vp, C.c_size_t, _vp]),
    "uaps_unet_ensemble_run": (_i, [_vp, C.c_size_t, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp, C.c_size_t, _vp, _vp, _vp, _vp,
                                    _vp]),
    "uaps_unet_ensemble_layer": (_i, [_i, _i, _i, _i, _vp, _vp, _vp, _vp]),
}

_lib: Optional[C.CDLL] = None


def exported_symbols() -> Sequence[str]:
    return tuple(_SIGNATURES)


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise loudly if it was never built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m uaps_b200.build` "
                "(or __graft_entry__.build()).  uaps_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the ABI and the binding diverge
            fn.restype, fn.argtypes = res, args
        if handle.uaps_abi_version() != ABI_VERSION:
            raise RuntimeError("libuaps_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().uaps_error_string(rc).decode()
        raise RuntimeError(f"{what} failed: {msg} (code {rc})")


class _NoSwitch:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_SWITCH = _NoSwitch()


def on_device(dev: torch.device):
    """Context that makes `dev` the current CUDA device -- a no-op object when it already is (one process per GPU:
    always), which saves the cudaGetDevice/cudaSetDevice pair of torch.cuda.device on ~1200 calls per iteration."""
    if dev.index is None or dev.index == torch.cuda.current_device():
        return _NO_SWITCH
    return torch.cuda.device(dev)


def stream_ptr() -> int:
    """Raw cudaStream_t the next launch goes to: torch's current stream -- taken once per training iteration when a
    StepContext is open (forward and autograd's backward of one iteration run on the stream that was current at its
    start), which saves a current_stream() lookup on each of the ~1150 launches."""
    sc = _stepctx._active
    if sc is not None and sc.stream is not None:
        return sc.stream
    return torch.cuda.current_stream().cuda_stream


def ptr_array(tensors: Sequence[Optional[torch.Tensor]]):
    """Host array of device pointers (``const float* const*``)."""
    arr = (_vp * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def float_array(vals: Sequence[float]):
    return (C.c_float * len(vals))(*[float(v) for v in vals])


def require_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("uaps_b200 kernels run on CUDA tensors only (no CPU fallback); got a "
                               f"{t.device} tensor")
