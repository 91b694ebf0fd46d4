"""ctypes binding of ``libmicronet_b200.so`` (the C-ABI in ``include/micronet_b200.h``).

There is no CPU fallback: if the shared library is missing, or a tensor is not on
a CUDA device, the call raises."""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmicronet_b200.so")

ACT_DOREFA, ACT_IAO, ACT_SIGN = 1, 2, 3


class ConvShape(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "batch", "in_c", "in_h", "in_w", "out_c", "ker_h", "ker_w", "stride_h", "stride_w",
        "pad_h", "pad_w", "dil_h", "dil_w", "groups")]


class ActQParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("bits", C.c_int32), ("qmin", C.c_int32), ("qmax", C.c_int32),
                ("q_type", C.c_int32), ("scale", C.c_void_p), ("zero_point", C.c_void_p),
                ("obs_min", C.c_void_p), ("obs_max", C.c_void_p)]


class PkPost(C.Structure):
    """mnb_pk_post: the consumer of a frozen-inference producer (its quantizer and operand plane)"""
    _fields_ = [("q", C.POINTER(ActQParams)), ("relu", C.c_int32), ("phase_split", C.c_int32), ("out_pk", C.c_void_p)]


class ConvOperands(C.Structure):
    _fields_ = [("a_codes", C.c_void_p), ("a_f32", C.c_void_p), ("a_offset", C.c_int32),
                ("a_offset_zp", C.c_void_p), ("a_scale", C.c_void_p), ("w_int", C.c_void_p),
                ("w_scale", C.c_void_p), ("w_f32", C.c_void_p), ("bias", C.c_void_p)]


_P, _I, _L, _D = C.c_void_p, C.c_int32, C.c_int64, C.c_double
_SHAPE, _ACTQ, _OPS = C.POINTER(ConvShape), C.POINTER(ActQParams), C.POINTER(ConvOperands)

# name -> (restype, argtypes); mirrors include/micronet_b200.h one to one
PROTOTYPES = {
    "mnb_version": (C.c_int, []),
    "mnb_last_error": (C.c_char_p, []),
    "mnb_launch_count": (_L, []),
    "mnb_act_quant_fwd": (C.c_int, [_P, _L, _ACTQ, _P, _P, _P, _P]),
    "mnb_act_quant_bwd": (C.c_int, [_P, _P, _L, _ACTQ, _P, _P]),
    "mnb_bn_fold_fwd": (C.c_int, [_P, _I, _I, _P, _P, _P, _P, _P, _D, _P, _P, _P]),
    "mnb_bn_fold_bwd": (C.c_int, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _D, _P, _P, _P]),
    "mnb_bn_fold_running": (C.c_int, [_P, _P, _P, _P, _I, _D, _I, _P]),
    "mnb_quant_add_fwd": (C.c_int, [_P, _P, _L, _ACTQ, _P, _P, _P, _I, _P]),
    "mnb_quant_add_bwd": (C.c_int, [_P, _P, _P, _L, _ACTQ, _P, _P, _P]),
    "mnb_observe_scratch_bytes": (_L, [_L, _I]),
    "mnb_iao_observe": (C.c_int, [_P, _L, _I, _I, _I, _D, _D, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "mnb_iao_update_qparams": (C.c_int, [_P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "mnb_dorefa_weight_fwd": (C.c_int, [_P, _L, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mnb_dorefa_weight_bwd": (C.c_int, [_P, _P, _L, _I, _P, _P, _P]),
    "mnb_wb_weight_fwd": (C.c_int, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mnb_wb_weight_bwd": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "mnb_iao_weight_fwd": (C.c_int, [_P, _L, _I, _I, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mnb_iao_weight_bwd": (C.c_int, [_P, _P, _P, _L, _I, _I, _P, _P]),
    "mnb_conv2d_fwd": (C.c_int, [_SHAPE, _OPS, _P, _P]),
    "mnb_conv2d_dgrad": (C.c_int, [_SHAPE, _P, _P, _P, _ACTQ, _P, _P]),
    "mnb_wgrad_scratch_bytes": (_L, [_SHAPE]),
    "mnb_conv2d_wgrad": (C.c_int, [_SHAPE, _P, _OPS, _P, _P, _P]),
    "mnb_channel_stats": (C.c_int, [_P, _I, _I, _I, _I, _P, _P, _P]),
    "mnb_channel_stats_bwd": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "mnb_bn_batch_stats": (C.c_int, [_P, _I, _I, _I, _D, _D, _P, _P, _P, _P, _P, _P]),
    "mnb_bn_sign_fwd": (C.c_int, [_P, _I, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P]),
    "mnb_bn_sign_bwd": (C.c_int, [_P, _P, _P, _I, _I, _I, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mnb_bn_sign_pool_fwd": (C.c_int, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P, _P]),
    "mnb_bn_sign_pool_bwd": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mnb_bn_sign_fwd_packed": (C.c_int, [_P, _I, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P, _P]),
    "mnb_fconv2d_fwd_tc": (C.c_int, [_SHAPE, _P, _P, _P, _P, _P, _P]),
    "mnb_fconv2d_wgrad_tc_scratch_bytes": (_L, [_SHAPE]),
    "mnb_fconv2d_wgrad_tc": (C.c_int, [_SHAPE, _P, _P, _P, _P, _P, _P]),
    "mnb_maxpool2d_fwd": (C.c_int, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "mnb_maxpool2d_bwd": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "mnb_adam_step": (C.c_int, [_P, _P, _P, _P, _L, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _I, _P]),
    "mnb_pk_act_bytes": (_L, [_I, _I, _I, _I, _I]),
    "mnb_pk_pack_act": (C.c_int, [_P, _I, _I, _I, _I, _ACTQ, _I, _P, _I, _P, _P, _P]),
    "mnb_bn_relu_quant_pack_fwd": (C.c_int, [_P, _I, _I, _I, _P, _P, _P, _P, _ACTQ, _I, _P, _P, _P]),
    "mnb_pk_pack_act_relu": (C.c_int, [_P, _I, _I, _I, _I, _ACTQ, _I, _P, _I, _I, _P, _P, _P]),
    "mnb_pk_conv_plan": (C.c_int, [_SHAPE, _I, _I, _I, _P]),
    "mnb_pk_wimage_bytes": (_L, [_SHAPE, _I, _I, _I]),
    "mnb_pk_pack_weight": (C.c_int, [_SHAPE, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mnb_pk_conv": (C.c_int, [_SHAPE, _I, _P, _I, _P, _I, _P, _P, C.c_float, _P, _P, C.c_float, _P, _P, _P]),
    "mnb_bn_sign_bwd_pack": (C.c_int, [_P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P, _P]),
    "mnb_bn_sign_pool_bwd_pack": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _I, _P, _P]),
    "mnb_pk_conv_post": (C.c_int, [_SHAPE, _P, _I, _P, _I, _P, _P, C.c_float, _P, _P, C.POINTER(PkPost), _P, _P]),
    "mnb_quant_add_pack_fwd": (C.c_int, [_P, _P, _I, _I, _I, _I, _ACTQ, _I, _P, C.POINTER(PkPost), _P]),
    "mnb_pk_wgrad_scratch_bytes": (_L, [_SHAPE, _I, _I]),
    "mnb_pk_wgrad": (C.c_int, [_SHAPE, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P]),
    "mnb_xnor_supported": (C.c_int, [_SHAPE]),
    "mnb_xnor_act_bytes": (_L, [_I, _I, _I, _I, _I]),
    "mnb_xnor_pack_act": (C.c_int, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "mnb_xnor_wimage_bytes": (_L, [_SHAPE]),
    "mnb_xnor_pack_weight": (C.c_int, [_SHAPE, _P, _P, _P]),
    "mnb_xnor_conv_fwd": (C.c_int, [_SHAPE, _P, _P, _P, _P, _P, _P]),
    "mnb_selftest_mma_rate": (C.c_int, [_I, _I, _I, _I, _I, _P, _P, _P]),
    "mnb_selftest_umma": (C.c_int, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "mnb_selftest_tma3d": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int32), _P, _P, _P]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"micronet_b200: {LIB_PATH} is missing - build it with `python -m micronet_b200.build` "
            "(there is no CPU / PyTorch fallback for the fake-quant hot path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().mnb_last_error().decode(errors="replace")
        kind = ValueError if rc < 0 else RuntimeError
        raise kind(f"micronet_b200.{what} failed (code {rc}): {msg}")


def ptr(t):
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "micronet_b200: the fake-quant engine runs on CUDA (sm_100a) tensors only; "
                "got a CPU tensor - there is deliberately no CPU fallback")


def require_f32(*tensors):
    """the C-ABI takes raw fp32 pointers: any other dtype would be misread silently"""
    for t in tensors:
        if t is not None and t.dtype != torch.float32:
            raise TypeError(f"micronet_b200: fp32 tensors only (the reference's QAT modules are fp32), got {t.dtype}")


def launch_count() -> int:
    return int(load().mnb_launch_count())


_errflags = {}


def tc_err_flag(device):
    """device int the tensor-core kernels set if a bounded pipeline wait ever times out"""
    key = (device.type, device.index)
    if key not in _errflags:
        _errflags[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return _errflags[key]


def tc_check(device=None):
    """synchronising check of the tensor-core error flag(s); raises if any kernel reported a timeout"""
    for key, flag in _errflags.items():
        code = int(flag.item())
        if code:
            raise RuntimeError(f"micronet_b200: tensor-core pipeline wait timed out (code {code}) on {key}")


E_UNSUPPORTED = -2
KEEP_DEBUG = False   # tests only: modules keep the fake-quantized weight of their last call
# packed-operand tensor-core family (mnb_pk.cu): "auto" = every fused-quantizer layer, every conv behind a binarizer and every
# conv the fp32 first-layer kernels (mnb_conv_fp32_tc.cu) do not take; "all" = every conv it supports, before those kernels;
# "off" = never (the generic kernels then run every conv: the reference arm of the tests)
PK_MODE = os.environ.get("MNB_PK", "auto")
# exact bf16 pieces per fp32 operand on the pk path (3 = exact 24-bit split; 2 = 16 bits, ~4e-6 relative)
PK_TERMS = int(os.environ.get("MNB_PK_TERMS", "3"))
# pieces of the fp32 operands of the BACKWARD convolutions (dy, the statistics conv's dpre, fp32 weights / inputs as their
# second operand).  Two pieces = 16 significand bits: gradient errors of ~3e-6 of the largest element (inside the 1e-5
# contract, every gradient check of the suite passes with margin) for 2/3 resp. 1/2 of the tensor-core work; nothing that
# decides an integer level depends on them.  The forward statistics conv keeps PK_TERMS (its mean / variance decide the
# quantized weight levels).  MNB_PK_TERMS_BWD=3 restores the exact split.
PK_TERMS_BWD = int(os.environ.get("MNB_PK_TERMS_BWD", "2"))

# bit-packed XNOR-popcount forward for wbwtab inference (mnb_xnor.cu): "auto" = the layers where it was measured to beat the
# tensor-core forward (functional.xnor_preferred), "all" = wherever it has cover, "off" = never
XNOR_MODE = os.environ.get("MNB_XNOR", "auto")

# fused BatchNorm + binarizer producers whose only reader takes the bf16 operand plane skip their fp32 output (fused.py
# _mark_plane_only); MNB_PLANE_ONLY=0 makes them write it again (e.g. to look at intermediate activations with hooks)
PLANE_ONLY = os.environ.get("MNB_PLANE_ONLY", "1") == "1"

_scratch = {}


def scratch(device, rows=1):
    """persistent zero-initialised scratch (block counters / histograms); kernels re-zero it."""
    lib = load()
    need = int(lib.mnb_observe_scratch_bytes(0, int(rows)))
    key = (device.type, device.index)
    buf = _scratch.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _scratch[key] = buf
    return buf
