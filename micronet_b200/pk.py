"""Python side of the packed-operand tensor-core family (``csrc/mnb_pk.cu``).

Every quantized conv of the QAT models runs here, from 1x1 grouped layers to ResNet-18's 512 -> 512 3x3 layers (weights
streamed, stride 2, 5x5 filters, 4x4 or 224x224 images); only the fp32 first layer (``mnb_conv_fp32_tc.cu``) and shapes
outside the cover (functional.QuantConv2dFn falls through to the generic kernels) do not:

    pack_act    fp32 NCHW -> bf16 term planes [t][b][c/8][h][w][8] (fake-quantize, or exact split of an fp32 tensor)
    pack_weight integer levels / fp32 weights -> the bf16 operand image of one (shape, mode)
    conv        TMA -> tcgen05.mma -> TMEM -> epilogue (forward: scale + bias; data gradient: STE mask)
    wgrad       the same boxes read as MN-major operands, split over the batch, deterministic reduction

Reference math: F.conv2d of the fake-quantized tensors (WB:186, DF:113, IAO:498/843/947) and ATen's
convolution_backward."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L

_plan_cache = {}


def _key(sh):
    return tuple(getattr(sh, f) for f, _ in sh._fields_)


def supported(sh, mode, terms_a, terms_w):
    """does mnb_pk_conv cover this (shape, mode)?  (host-only plan query, cached)"""
    k = ("c", _key(sh), mode, terms_a, terms_w)
    if k not in _plan_cache:
        _plan_cache[k] = L.load().mnb_pk_conv_plan(C.byref(sh), mode, terms_a, terms_w, None) == 0
    return _plan_cache[k]


def wgrad_supported(sh, terms_dy, terms_x):
    k = ("w", _key(sh), terms_dy, terms_x)
    if k not in _plan_cache:
        _plan_cache[k] = int(L.load().mnb_pk_wgrad_scratch_bytes(C.byref(sh), terms_dy, terms_x))
    return _plan_cache[k] >= 0


def pack_act(x, qp, terms, ch_scale=None, phase_split=False, want_bits=False, relu=False):
    """-> (planes u8[terms * B * ceil(C/8) * H * W * 16], bits8 u8[B, ceil(C/8), H, W] or None)"""
    lib = L.load()
    b, c, h, w = x.shape
    nbytes = int(lib.mnb_pk_act_bytes(b, c, h, w, terms))
    out = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    bits = None
    if qp is not None and want_bits:
        bits = torch.empty((b, (c + 7) // 8, h, w), dtype=torch.uint8, device=x.device)
    L.check(lib.mnb_pk_pack_act_relu(x.data_ptr(), b, c, h, w, None if qp is None else C.byref(qp), terms, L.ptr(ch_scale),
                                     1 if phase_split else 0, 1 if relu else 0, out.data_ptr(), L.ptr(bits), L.stream()),
            "pk_pack_act")
    return out, bits


def pack_weight(sh, mode, terms_a, terms_w, w_int=None, w_f32=None, kzero=None):
    lib = L.load()
    nbytes = int(lib.mnb_pk_wimage_bytes(C.byref(sh), mode, terms_a, terms_w))
    if nbytes < 0:
        raise ValueError("micronet_b200.pk: shape outside the cover of the packed-operand convolution")
    dev = (w_int if w_int is not None else w_f32).device
    img = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    L.check(lib.mnb_pk_pack_weight(C.byref(sh), mode, terms_a, terms_w, L.ptr(w_int), L.ptr(w_f32), L.ptr(kzero),
                                   img.data_ptr(), L.stream()), "pk_pack_weight")
    return img


def conv(sh, mode, a_pk, terms_a, w_img, terms_w, out, n_scale=None, a_scale=None, a_scale_const=1.0, bias=None,
         bits8=None, gain=1.0):
    lib = L.load()
    return lib.mnb_pk_conv(C.byref(sh), mode, a_pk.data_ptr(), terms_a, w_img.data_ptr(), terms_w, L.ptr(n_scale),
                           L.ptr(a_scale), float(a_scale_const), L.ptr(bias), L.ptr(bits8), float(gain), out.data_ptr(),
                           L.tc_err_flag(out.device).data_ptr(), L.stream())


def consumer_plane(b, c, h, w, device):
    """empty operand plane (one bf16 piece) of a conv that reads a [b, c, h, w] activation"""
    return torch.empty(int(L.load().mnb_pk_act_bytes(b, c, h, w, 1)), dtype=torch.uint8, device=device)


def conv_post(sh, a_pk, terms_a, w_img, terms_w, out, post_qp, post_plane, post_relu, post_split, n_scale=None, a_scale=None,
              a_scale_const=1.0, bias=None):
    """forward conv whose epilogue also writes the consumer's operand plane (frozen inference graphs); out may be None"""
    lib = L.load()
    post = L.PkPost(C.pointer(post_qp), 1 if post_relu else 0, 1 if post_split else 0, post_plane.data_ptr())
    return lib.mnb_pk_conv_post(C.byref(sh), a_pk.data_ptr(), terms_a, w_img.data_ptr(), terms_w, L.ptr(n_scale), L.ptr(a_scale),
                                float(a_scale_const), L.ptr(bias), L.ptr(out), C.byref(post),
                                L.tc_err_flag(a_pk.device).data_ptr(), L.stream())


def wgrad(sh, dy_pk, terms_dy, x_pk, terms_x, dw, a_scale=None, kdiv=None):
    lib = L.load()
    nbytes = int(lib.mnb_pk_wgrad_scratch_bytes(C.byref(sh), terms_dy, terms_x))
    if nbytes < 0:
        return L.E_UNSUPPORTED
    ws = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dw.device)
    return lib.mnb_pk_wgrad(C.byref(sh), dy_pk.data_ptr(), terms_dy, x_pk.data_ptr(), terms_x, L.ptr(a_scale),
                            L.ptr(kdiv), dw.data_ptr(), ws.data_ptr(), L.tc_err_flag(dw.device).data_ptr(), L.stream())
