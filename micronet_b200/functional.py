"""autograd.Function wrappers around the C-ABI kernels.

Each Function mirrors one autograd node (or a fused chain of nodes) of the
reference's forward path; the math each kernel implements is documented in
``include/micronet_b200.h`` with the reference file:line it replaces."""
from __future__ import annotations

import ctypes as C

import torch
from torch.autograd import Function

from . import _lib as L


# --------------------------------------------------------------------------
# optional per-launch device timing of the conv kernels (bench.py's roofline leg)
# --------------------------------------------------------------------------
class KernelTimer:
    """records a CUDA-event pair on the launching (current) stream around each conv kernel call"""

    def __init__(self):
        self.records = []  # (kind, shape tuple, start event, end event)

    def run(self, kind, sh, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = fn()
        b.record()
        self.records.append((kind, tuple(getattr(sh, f) for f, _ in sh._fields_), a, b))
        return rc

    def summary(self):
        """{(kind, shape): [ms, ...]} — call after torch.cuda.synchronize()"""
        out = {}
        for kind, shape, a, b in self.records:
            out.setdefault((kind, shape), []).append(a.elapsed_time(b))
        return out


TIMER = None  # set to a KernelTimer to enable


def _timed(kind, sh, fn):
    return fn() if TIMER is None else TIMER.run(kind, sh, fn)


# --------------------------------------------------------------------------
# activation quantizer description
# --------------------------------------------------------------------------
class ActSpec:
    """Which activation fake-quantizer to run and where its device-resident
    parameters live (tensors are the module's registered buffers)."""

    __slots__ = ("mode", "bits", "qmin", "qmax", "q_type", "scale", "zero_point", "obs_min", "obs_max")

    def __init__(self, mode, bits=8, qmin=0, qmax=255, q_type=0, scale=None, zero_point=None,
                 obs_min=None, obs_max=None):
        self.mode, self.bits, self.qmin, self.qmax, self.q_type = mode, bits, qmin, qmax, q_type
        self.scale, self.zero_point, self.obs_min, self.obs_max = scale, zero_point, obs_min, obs_max

    def struct(self):
        return L.ActQParams(self.mode, self.bits, self.qmin, self.qmax, self.q_type, L.ptr(self.scale),
                            L.ptr(self.zero_point), L.ptr(self.obs_min), L.ptr(self.obs_max))

    def frozen(self):
        """copy with private clones of the device scalars: what backward must see is the forward-time scale / range
        (the reference uses self.scale.clone(), IAO:228-239), not whatever a later forward of the module wrote"""
        if self.mode != L.ACT_IAO:
            return self
        snap = torch.cat([self.scale.reshape(1), self.zero_point.reshape(1), self.obs_min.reshape(1), self.obs_max.reshape(1)])
        return ActSpec(self.mode, self.bits, self.qmin, self.qmax, self.q_type, snap[0:1], snap[1:2], snap[2:3], snap[3:4])

    # decoding of the u8 codes: effective integer e = code + offset (+ zero_point), value = e * scale
    @property
    def code_offset(self):
        if self.mode == L.ACT_IAO:
            return self.qmin
        if self.mode == L.ACT_SIGN:
            return -1
        return 0


def _dorefa_scale_tensor(bits, device, _cache={}):
    key = (bits, device.type, device.index)
    if key not in _cache:
        # Python double 1/(2^a-1), cast to fp32 exactly as ATen does for `tensor / python_float`
        _cache[key] = torch.tensor([1.0 / float(2 ** bits - 1)], dtype=torch.float32, device=device)
    return _cache[key]


def act_quant_raw(x, spec: ActSpec, want_codes, want_bits, want_xq):
    """run the activation quantizer kernel; returns (codes, pass_bits, xq)"""
    L.require_cuda(x)
    lib = L.load()
    x = x.contiguous()
    n = x.numel()
    codes = torch.empty(x.shape, dtype=torch.uint8, device=x.device) if want_codes else None
    bits = torch.empty((n + 31) // 32, dtype=torch.int32, device=x.device) if want_bits else None
    xq = torch.empty_like(x) if want_xq else None
    qp = spec.struct()
    L.check(lib.mnb_act_quant_fwd(x.data_ptr(), n, C.byref(qp), L.ptr(codes), L.ptr(bits), L.ptr(xq),
                                  L.stream()), "act_quant_fwd")
    return codes, bits, xq


class ActQuantFn(Function):
    """standalone fake-quant of an activation tensor (reference: ActivationQuantizer /
    Quantizer.forward returning the dequantized tensor)."""

    @staticmethod
    def forward(ctx, x, spec: ActSpec):
        _, bits, xq = act_quant_raw(x, spec, False, ctx.needs_input_grad[0], True)
        ctx.spec, ctx.bits = (spec.frozen() if ctx.needs_input_grad[0] else spec), bits
        return xq

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        g = g.contiguous()
        dx = torch.empty_like(g)
        qp = ctx.spec.struct()
        L.check(lib.mnb_act_quant_bwd(g.data_ptr(), ctx.bits.data_ptr(), g.numel(), C.byref(qp),
                                      dx.data_ptr(), L.stream()), "act_quant_bwd")
        return dx, None


class QuantAddFn(Function):
    """IAO QuantAdd (IAO:1441-1498): Q(res) + Q(shortcut) with the shared quantizer, one kernel each way"""

    @staticmethod
    def forward(ctx, a, b, spec: ActSpec, relu=False):
        L.require_cuda(a, b)
        lib = L.load()
        a, b = a.contiguous(), b.contiguous()
        assert a.shape == b.shape, "QuantAdd: operand shapes differ"
        n = a.numel()
        out = torch.empty_like(a)
        words = (n + 31) // 32
        ba = torch.empty(words, dtype=torch.int32, device=a.device) if ctx.needs_input_grad[0] else None
        bb = torch.empty(words, dtype=torch.int32, device=a.device) if ctx.needs_input_grad[1] else None
        qp = spec.struct()
        assert not (relu and (ba is not None or bb is not None)), "the folded ReLU is an inference-only fusion"
        L.check(lib.mnb_quant_add_fwd(a.data_ptr(), b.data_ptr(), n, C.byref(qp), out.data_ptr(), L.ptr(ba), L.ptr(bb),
                                      1 if relu else 0, L.stream()), "quant_add_fwd")
        ctx.spec, ctx.ba, ctx.bb = spec.frozen() if (ba is not None or bb is not None) else spec, ba, bb
        return out

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        g = g.contiguous()
        da = torch.empty_like(g) if ctx.ba is not None else None
        db = torch.empty_like(g) if ctx.bb is not None else None
        qp = ctx.spec.struct()
        L.check(lib.mnb_quant_add_bwd(g.data_ptr(), L.ptr(ctx.ba), L.ptr(ctx.bb), g.numel(), C.byref(qp), L.ptr(da),
                                      L.ptr(db), L.stream()), "quant_add_bwd")
        return da, db, None, None


# --------------------------------------------------------------------------
# weight quantizers: return (wq fp32, w_int i16, w_scale f32[K])
# --------------------------------------------------------------------------
class DorefaWeightFn(Function):
    @staticmethod
    def forward(ctx, w, w_bits):
        L.require_cuda(w)
        lib = L.load()
        w = w.contiguous()
        n, k = w.numel(), w.shape[0]
        wq = torch.empty_like(w)
        w_int = torch.empty(w.shape, dtype=torch.int16, device=w.device)
        w_scale = torch.empty(k, dtype=torch.float32, device=w.device)
        aux = torch.empty(n + 4, dtype=torch.float32, device=w.device)
        L.check(lib.mnb_dorefa_weight_fwd(w.data_ptr(), n, k, w_bits, w_int.data_ptr(), w_scale.data_ptr(),
                                          wq.data_ptr(), aux.data_ptr(), L.scratch(w.device).data_ptr(),
                                          L.stream()), "dorefa_weight_fwd")
        ctx.aux, ctx.w_bits = aux, w_bits
        ctx.mark_non_differentiable(w_int, w_scale)
        return wq, w_int, w_scale

    @staticmethod
    def backward(ctx, g, _gi, _gs):
        lib = L.load()
        g = g.contiguous()
        dw = torch.empty_like(g)
        L.check(lib.mnb_dorefa_weight_bwd(g.data_ptr(), ctx.aux.data_ptr(), g.numel(), ctx.w_bits,
                                          dw.data_ptr(), L.scratch(g.device).data_ptr(), L.stream()),
                "dorefa_weight_bwd")
        return dw, None


class WbWeightFn(Function):
    """wbwtab binary / ternary weights.  W == 2 mutates ``w`` in place (WB:98-102)."""

    @staticmethod
    def forward(ctx, w, W):
        L.require_cuda(w)
        lib = L.load()
        assert w.is_contiguous() and w.dim() == 4
        k, cpg, khw = w.shape[0], w.shape[1], w.shape[2] * w.shape[3]
        wq = torch.empty_like(w)
        w_int = torch.empty(w.shape, dtype=torch.int16, device=w.device)
        w_scale = torch.empty(k, dtype=torch.float32, device=w.device)
        aux = torch.empty(3 * k, dtype=torch.float32, device=w.device)
        L.check(lib.mnb_wb_weight_fwd(w.data_ptr(), k, cpg, khw, W, w_int.data_ptr(), w_scale.data_ptr(),
                                      wq.data_ptr(), aux.data_ptr(), L.stream()), "wb_weight_fwd")
        ctx.w, ctx.aux, ctx.W = w.detach(), aux, W  # gradient is taken at the (mutated) parameter values
        ctx.mark_non_differentiable(w_int, w_scale)
        return wq, w_int, w_scale

    @staticmethod
    def backward(ctx, g, _gi, _gs):
        lib = L.load()
        g = g.contiguous()
        w = ctx.w
        dw = torch.empty_like(g)
        L.check(lib.mnb_wb_weight_bwd(g.data_ptr(), w.data_ptr(), ctx.aux.data_ptr(), w.shape[0], w.shape[1],
                                      w.shape[2] * w.shape[3], ctx.W, dw.data_ptr(), L.stream()),
                "wb_weight_bwd")
        return dw, None


class IaoWeightFn(Function):
    """IAO fake-quant of a weight tensor with (already refreshed) per-row or per-layer qparams."""

    @staticmethod
    def forward(ctx, w, scale, zero_point, obs_min, obs_max, q_type, qmin, qmax):
        L.require_cuda(w)
        lib = L.load()
        w = w.contiguous()
        n, k, rows = w.numel(), w.shape[0], scale.numel()
        wq = torch.empty_like(w)
        w_int = torch.empty(w.shape, dtype=torch.int16, device=w.device)
        w_scale = torch.empty(k, dtype=torch.float32, device=w.device)
        keep = torch.empty(w.shape, dtype=torch.uint8, device=w.device)
        L.check(lib.mnb_iao_weight_fwd(w.data_ptr(), n, k, rows, scale.data_ptr(), zero_point.data_ptr(),
                                       obs_min.data_ptr(), obs_max.data_ptr(), q_type, qmin, qmax,
                                       w_int.data_ptr(), w_scale.data_ptr(), wq.data_ptr(), keep.data_ptr(),
                                       L.stream()), "iao_weight_fwd")
        ctx.keep, ctx.scale, ctx.k, ctx.rows = keep, scale, k, rows
        ctx.mark_non_differentiable(w_int, w_scale)
        return wq, w_int, w_scale

    @staticmethod
    def backward(ctx, g, _gi, _gs):
        lib = L.load()
        g = g.contiguous()
        dw = torch.empty_like(g)
        L.check(lib.mnb_iao_weight_bwd(g.data_ptr(), ctx.keep.data_ptr(), ctx.scale.data_ptr(), g.numel(),
                                       ctx.k, ctx.rows, dw.data_ptr(), L.stream()), "iao_weight_bwd")
        return (dw,) + (None,) * 7


# --------------------------------------------------------------------------
# the fake-quantized convolution
# --------------------------------------------------------------------------
def _shape_struct(x_shape, w_shape, stride, padding, dilation, groups):
    b, c, h, w = x_shape
    k, _, r, s = w_shape
    return L.ConvShape(b, c, h, w, k, r, s, stride[0], stride[1], padding[0], padding[1],
                       dilation[0], dilation[1], groups)


def _out_hw(sh: L.ConvShape):
    p = (sh.in_h + 2 * sh.pad_h - sh.dil_h * (sh.ker_h - 1) - 1) // sh.stride_h + 1
    q = (sh.in_w + 2 * sh.pad_w - sh.dil_w * (sh.ker_w - 1) - 1) // sh.stride_w + 1
    return p, q


def channel_sums(x4):
    """sum over (B, H, W) of a [B, C, H, W] tensor -> [C] (bias gradient)."""
    lib = L.load()
    b, c = x4.shape[0], x4.shape[1]
    hw = x4.numel() // (b * c)
    out = torch.empty(2 * c, dtype=torch.float32, device=x4.device)
    L.check(lib.mnb_channel_stats(x4.data_ptr(), b, c, hw, 0, out.data_ptr(),
                                  L.scratch(x4.device, c).data_ptr(), L.stream()), "channel_stats")
    return out[:c]



def materialized(t):
    """the values of a producer output: ``t`` itself, or - for a plane-only output of a fused BatchNorm + binarizer (its fp32
    storage was never written) - the +-1 tensor rebuilt from the bf16 operand plane [b][c/8][h][w][8].  Plumbing for tests,
    hooks and convs outside the packed-operand cover; the training step never calls it."""
    if not getattr(t, "_mnb_plane_only", False):
        return t
    b, c, h, w = t.shape
    plane = t._mnb_pk_pm1.view(torch.bfloat16).view(b, c // 8, h, w, 8)
    return plane.permute(0, 1, 4, 2, 3).reshape(b, c, h, w).float()


def xnor_preferred(sh, has_plane):
    """MNB_XNOR=auto: take the XNOR-popcount forward for this wbwtab inference layer?  Decided from the layer-by-layer
    measurement of harness/xnor_probe.py on B200 (profiles/r2_xnor_vs_tc.md, NIN-GC layers at batch 256):

    * the two convolution kernels tie within ~7 % on the 1x1 layers (29 - 87 us vs 27 - 81 us) and split the 3x3 layers
      (102 vs 83 us, 56 vs 58 us): both are dominated by the fp32 output they write, and B200's popc pipe (16 lanes / clk /
      SM) gives the bit kernel no arithmetic edge over tcgen05 on +-1 operands;
    * the operand it reads is 16 x smaller (1 bit vs one bf16 per activation): packing it from an fp32 tensor costs 11 - 50 us
      against 25 - 156 us for the bf16 plane, so a layer that has to pack its own input is 1.08 - 1.79 x faster end to end.

    Hence: XNOR when the layer packs its own operand (no producer-written plane came with x), the tensor-core forward when a
    fused BatchNorm + binarizer already wrote the bf16 plane (the pack pass is free there)."""
    return not has_plane


def _pk_terms(spec, w_int, pm1=False):
    """(terms of the activation operand, terms of the weight operand) on the packed-operand path; ``pm1``: the raw input is
    known to hold only +-1 (output of a binarizer): one bf16 piece is exact"""
    T = L.PK_TERMS
    if spec is None:
        ta = 1 if pm1 else T
    else:
        ta = 2 if (spec.mode == L.ACT_IAO and spec.q_type == 1) else 1   # asymmetric: |level + zero_point| may exceed 256
    return ta, (1 if w_int is not None else T)


def _pk_forward(ctx, x, wq, bias, w_int, w_scale, spec, sh, y, need_dx, prepacked=None, pre_relu=False, pm1=False):
    """forward on the packed-operand tensor-core family; returns False when the shape is outside its cover.
    ``prepacked``: the operand plane a fused producer (fused.BNReluQuantFn) already wrote - x itself holds no data then."""
    from . import pk as PK
    ta, tw = _pk_terms(spec, w_int, pm1)
    if not PK.supported(sh, 0, ta, tw):
        return False
    # the backward of a layer stays in the family its forward ran in (saved operands are packed): check its cover now
    Tb = min(L.PK_TERMS, L.PK_TERMS_BWD)
    if need_dx and not PK.supported(sh, 1, Tb, 1 if w_int is not None else Tb):
        return False
    if ctx.needs_input_grad[1] and not PK.wgrad_supported(sh, Tb, min(ta, Tb)):
        return False
    qp = spec.struct() if spec is not None else None
    split = sh.stride_h == 2
    if prepacked is not None:
        x_pk, bits8 = prepacked, None      # the producer keeps the STE mask for its own backward
    else:
        x_pk, bits8 = PK.pack_act(x, qp, ta, phase_split=split, want_bits=need_dx, relu=pre_relu)
    # frozen (inference) modules hang a dict on their cached weight tensor: the packed image is then built once
    src = w_int if w_int is not None else wq
    cache = getattr(src, "_mnb_pk_cache", None)
    ckey = (PK._key(sh), ta, tw)
    w_img = cache.get(ckey) if cache is not None else None
    if w_img is None:
        w_img = PK.pack_weight(sh, 0, ta, tw, w_int=w_int, w_f32=None if w_int is not None else wq)
        if cache is not None:
            cache[ckey] = w_img
    a_scale, a_const = None, 1.0
    if spec is not None:
        if spec.mode == L.ACT_IAO:
            # backward must see the forward-time scale (the reference clones it too); no clone needed without autograd
            a_scale = spec.scale.clone() if (need_dx or ctx.needs_input_grad[1]) else spec.scale
        elif spec.mode == L.ACT_DOREFA:
            a_const = 1.0 / float(2 ** spec.bits - 1)
    rc = _timed("fwd_pk", sh, lambda: PK.conv(sh, 0, x_pk, ta, w_img, tw, y, n_scale=w_scale if w_int is not None else None,
                                              a_scale=a_scale, a_scale_const=a_const, bias=bias))
    if rc == L.E_UNSUPPORTED:
        return False
    L.check(rc, "pk_conv fwd")
    ctx.pk = True
    ctx.pk_x, ctx.pk_ta, ctx.pk_bits8, ctx.pk_a_scale, ctx.pk_prepacked = x_pk, ta, bits8, a_scale, prepacked is not None
    return True


def _pk_backward(ctx, dy):
    """data and weight gradients of a layer whose forward ran on the packed-operand path"""
    from . import pk as PK
    sh, spec = ctx.sh, ctx.spec
    T = min(L.PK_TERMS, L.PK_TERMS_BWD)     # pieces of dy and of an fp32 second operand (see _lib.PK_TERMS_BWD)
    int_w = ctx.w_int is not None
    need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
    # dy is packed once for both gradients; the data gradient wants the per-channel weight scale folded in (it sits on
    # the reduction dimension there), the weight gradient divides it out again (mnb_pk_wgrad's kdiv)
    fold = int_w and need_dx
    pre = getattr(dy, "_mnb_pk_dy", None)     # written by the consumer's fused BatchNorm backward (fused.BNSignFn): dy holds no data
    if pre is not None:
        if pre[1] != T or (pre[2] is not None) != fold:
            raise RuntimeError("micronet_b200: packed gradient operand does not match this layer's backward configuration")
        dy_pk = pre[0]
    else:
        dy_pk, _ = PK.pack_act(dy, None, T, ch_scale=ctx.w_scale if fold else None)
    dx = dwq = None
    if need_dx:
        tw = 1 if int_w else T
        w_img = PK.pack_weight(sh, 1, T, tw, w_int=ctx.w_int, w_f32=None if int_w else ctx.wq,
                               kzero=ctx.w_scale if int_w else None)
        dx = torch.empty((sh.batch, sh.in_c, sh.in_h, sh.in_w), dtype=torch.float32, device=dy.device)
        gain = 0.1 if (spec is not None and spec.mode == L.ACT_DOREFA) else 1.0
        # a fused producer applies the STE mask itself (it owns the mask bits): plain data gradient times the quantizer's gain
        plain_gain = gain if ctx.pk_prepacked else 1.0
        L.check(_timed("dgrad_pk", sh, lambda: PK.conv(sh, 1, dy_pk, T, w_img, tw, dx, bits8=ctx.pk_bits8, gain=gain,
                                                       a_scale_const=plain_gain)), "pk_conv dgrad")
    if need_dw:
        dwq = torch.empty_like(ctx.wq)
        a_scale = None
        if spec is not None:
            a_scale = ctx.pk_a_scale if spec.mode == L.ACT_IAO else _dorefa_scale_tensor(spec.bits, dy.device)
        tx = min(ctx.pk_ta, T)     # a 3-piece saved input contributes its two leading pieces
        L.check(_timed("wgrad_pk", sh, lambda: PK.wgrad(sh, dy_pk, T, ctx.pk_x, tx, dwq, a_scale=a_scale,
                                                        kdiv=ctx.w_scale if fold else None)), "pk_wgrad")
    return dx, dwq


class QuantConv2dFn(Function):
    """y = conv2d(Q_a(x), wq, bias) with the activation quantizer fused on the input side
    and the clip-STE fused into dgrad.  ``spec`` None => x is used as fp32 (wbwtab, a_bits=32)."""

    @staticmethod
    def forward(ctx, x, wq, bias, w_int, w_scale, spec, stride, padding, dilation, groups, pre_relu=False, no_grad=False):
        L.require_cuda(x, wq)
        assert not (pre_relu and any(ctx.needs_input_grad)), "the folded ReLU is an inference-only fusion"
        lib = L.load()
        x = x.contiguous()
        wq = wq.contiguous()
        sh = _shape_struct(x.shape, wq.shape, stride, padding, dilation, groups)
        p, q = _out_hw(sh)
        y = torch.empty((x.shape[0], wq.shape[0], p, q), dtype=torch.float32, device=x.device)
        codes = bits = None
        a_scale = None
        if spec is not None and spec.mode != L.ACT_SIGN:
            a_scale = spec.scale if spec.mode == L.ACT_IAO else _dorefa_scale_tensor(spec.bits, x.device)
        done = False
        ctx.pk = False
        if (L.XNOR_MODE != "off" and spec is None and w_int is not None and getattr(x, "_mnb_pm1", False)
                and (no_grad or not any(ctx.needs_input_grad[:3])) and x.dtype == torch.float32 and not pre_relu):
            # wbwtab inference forward on +-1 activations: bit-packed XNOR-popcount kernel where it was measured to beat the
            # tensor-core forward (north_star; table: profiles/r2_xnor_vs_tc.md).  Same integer sums, same fmaf epilogue:
            # bit-identical to the packed-operand path.  Training steps never come here (their backward multiplies real-valued
            # gradients and wants the bf16 operand plane the forward already read).
            from . import xnor as XN
            if XN.supported(sh) and (L.XNOR_MODE == "all" or xnor_preferred(sh, getattr(x, "_mnb_pk_pm1", None) is not None)):
                a_bits = XN.pack_act(materialized(x), groups)
                rc = _timed("fwd_xnor", sh, lambda: XN.conv(sh, a_bits, XN.pack_weight(sh, w_int), y, alpha=w_scale, bias=bias))
                if rc == 0:
                    done = True
                elif rc != L.E_UNSUPPORTED:
                    L.check(rc, "xnor_conv_fwd")
        pkq = getattr(x, "_mnb_pk_q", None)   # operand plane written by a fused BN + ReLU + quantizer producer
        if pkq is not None and not done:
            if spec is None or spec.mode != L.ACT_DOREFA or spec.bits != pkq[1] or w_int is None:
                raise RuntimeError("micronet_b200: a fused producer's packed output reached a conv with another quantizer")
            done = _pk_forward(ctx, x, wq, bias, w_int, w_scale, spec, sh, y, ctx.needs_input_grad[0], prepacked=pkq[0])
            if not done:
                raise RuntimeError("micronet_b200: fused producer output in front of a conv outside the packed-operand cover")
        if (not done and L.PK_MODE != "off" and x.dtype == torch.float32 and (L.PK_MODE == "all" or spec is not None)
                and not getattr(x, "_mnb_plane_only", False)):
            done = _pk_forward(ctx, x, wq, bias, w_int, w_scale, spec, sh, y, ctx.needs_input_grad[0], pre_relu=pre_relu)
        if (not done and L.PK_MODE != "off" and spec is None and x.dtype == torch.float32 and getattr(x, "_mnb_pm1", False)
                and not pre_relu):
            # conv behind a binarizer (a wbwtab layer, or with fp32 weights the 10-way head, fused.EnginePmConv2d): the +-1
            # input is ONE exact bf16 piece.  With the plane a fused BatchNorm + binarizer wrote (fused.BNSignFn) the layer is
            # pure TMA -> MMA, without it the layer packs its own input
            plane = getattr(x, "_mnb_pk_pm1", None)
            if plane is not None and plane.numel() != x.numel() * 2:
                plane = None
            done = _pk_forward(ctx, x, wq, bias, w_int, w_scale, None, sh, y, ctx.needs_input_grad[0], prepacked=plane,
                               pm1=True)
        if not done and getattr(x, "_mnb_plane_only", False):
            x = materialized(x)   # outside the packed-operand cover (rare): the kernels below read the fp32 values
        if not done and pre_relu:
            x = torch.relu(x)     # outside the packed-operand cover: the folded ReLU as its own pass
        ctx.fconv = False
        if not done and spec is None and x.dtype == torch.float32:
            # un-quantized input with few channels (first layer): fp32-accurate im2col conv on the tensor cores
            rc = _timed("fconv_fwd_tc", sh, lambda: lib.mnb_fconv2d_fwd_tc(
                C.byref(sh), x.data_ptr(), wq.data_ptr(), L.ptr(bias), y.data_ptr(),
                L.tc_err_flag(x.device).data_ptr(), L.stream()))
            if rc == 0:
                done = ctx.fconv = True
            elif rc != L.E_UNSUPPORTED:
                L.check(rc, "fconv2d_fwd_tc")
        if not done and L.PK_MODE != "off" and x.dtype == torch.float32:
            done = _pk_forward(ctx, x, wq, bias, w_int, w_scale, spec, sh, y, ctx.needs_input_grad[0])
        if not done:
            ops = L.ConvOperands()
            if spec is not None:
                codes, bits, _ = act_quant_raw(x, spec, True, ctx.needs_input_grad[0], False)
                ops.a_codes = codes.data_ptr()
                ops.a_offset = spec.code_offset
                ops.a_offset_zp = L.ptr(spec.zero_point) if spec.mode == L.ACT_IAO else None
                ops.a_scale = L.ptr(a_scale)
            else:
                ops.a_f32 = x.data_ptr()
            if codes is not None and w_int is not None:
                ops.w_int, ops.w_scale = w_int.data_ptr(), w_scale.data_ptr()
            else:
                ops.w_f32 = wq.data_ptr()
            ops.bias = L.ptr(bias)
            L.check(_timed("fwd", sh, lambda: lib.mnb_conv2d_fwd(C.byref(sh), C.byref(ops), y.data_ptr(), L.stream())),
                    "conv2d_fwd")
        if spec is not None and not ctx.pk and (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]):
            spec = spec.frozen()   # backward re-quantizes / masks with the forward-time parameters
            if spec.mode == L.ACT_IAO:
                a_scale = spec.scale
        ctx.sh, ctx.spec, ctx.a_scale = sh, spec, a_scale
        ctx.codes, ctx.bits = codes, bits
        ctx.x = x if (not ctx.pk and codes is None) else None   # fp32 input of the generic / tcfp32 weight gradient
        ctx.wq = wq
        ctx.w_int, ctx.w_scale = (w_int, w_scale) if w_int is not None else (None, None)
        ctx.has_bias = bias is not None
        if ctx.pk and spec is None and w_int is not None and ctx.needs_input_grad[1]:
            # a fused BatchNorm + binarizer consuming y may write this layer's gradient operand itself (fused.BNSignFn)
            y._mnb_pk_conv = (w_scale if ctx.needs_input_grad[0] else None, min(L.PK_TERMS, L.PK_TERMS_BWD))
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        # a fused BatchNorm+binarize consumer already reduced its dx (= this dy) over (B, H, W): fused.BNSignFn
        presummed = getattr(dy, "_mnb_channel_sum", None)
        dy = dy.contiguous()
        sh, spec = ctx.sh, ctx.spec
        dx = dwq = db = None
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = presummed if presummed is not None and presummed.numel() == dy.shape[1] else channel_sums(dy)
        if ctx.pk:
            dx, dwq = _pk_backward(ctx, dy)
            return dx, dwq, db, None, None, None, None, None, None, None, None, None
        if ctx.needs_input_grad[0]:
            dx = torch.empty((sh.batch, sh.in_c, sh.in_h, sh.in_w), dtype=torch.float32, device=dy.device)
            qp = spec.struct() if spec is not None else None
            bits_ptr = ctx.bits.data_ptr() if spec is not None else None
            L.check(_timed("dgrad", sh, lambda: lib.mnb_conv2d_dgrad(
                C.byref(sh), dy.data_ptr(), ctx.wq.data_ptr(), bits_ptr, None if qp is None else C.byref(qp),
                dx.data_ptr(), L.stream())), "conv2d_dgrad")
        if ctx.needs_input_grad[1]:
            dwq = torch.empty_like(ctx.wq)
            fbytes = int(lib.mnb_fconv2d_wgrad_tc_scratch_bytes(C.byref(sh))) if ctx.fconv else -1
            if fbytes >= 0:
                ws = torch.empty(max(fbytes, 4), dtype=torch.uint8, device=dy.device)
                L.check(_timed("fconv_wgrad_tc", sh, lambda: lib.mnb_fconv2d_wgrad_tc(
                    C.byref(sh), dy.data_ptr(), ctx.x.data_ptr(), dwq.data_ptr(), ws.data_ptr(),
                    L.tc_err_flag(dy.device).data_ptr(), L.stream())), "fconv2d_wgrad_tc")
            else:
                ops = L.ConvOperands()
                if ctx.codes is not None:
                    ops.a_codes = ctx.codes.data_ptr()
                    ops.a_offset = spec.code_offset
                    ops.a_offset_zp = L.ptr(spec.zero_point) if spec.mode == L.ACT_IAO else None
                    ops.a_scale = L.ptr(ctx.a_scale)
                else:
                    ops.a_f32 = ctx.x.data_ptr()
                nbytes = int(lib.mnb_wgrad_scratch_bytes(C.byref(sh)))
                ws = torch.empty(max(nbytes, 4), dtype=torch.uint8, device=dy.device)
                L.check(_timed("wgrad", sh, lambda: lib.mnb_conv2d_wgrad(
                    C.byref(sh), dy.data_ptr(), C.byref(ops), dwq.data_ptr(), ws.data_ptr(), L.stream())),
                    "conv2d_wgrad")
        return dx, dwq, db, None, None, None, None, None, None, None, None, None


def quant_conv2d(x, wq, bias, w_int, w_scale, spec, stride, padding, dilation, groups, pre_relu=False):
    # (autograd runs a Function's forward with grad mode off and needs_input_grad ignores torch.no_grad(): whether this call
    # will ever be differentiated is only known out here)
    return QuantConv2dFn.apply(x, wq, bias, w_int, w_scale, spec, tuple(stride), tuple(padding),
                               tuple(dilation), groups, pre_relu, not torch.is_grad_enabled())


# --------------------------------------------------------------------------
# transposed convolution (IAO.QuantConvTranspose2d, IAO:510-636)
# --------------------------------------------------------------------------
def _pk_plain(sh, mode, a, w, out, T):
    """fp32 x fp32 convolution (mode 0) / data gradient (mode 1) of shape ``sh`` on the packed-operand tensor-core family:
    both operands as T exact bf16 pieces.  False when the shape is outside its cover."""
    from . import pk as PK
    if L.PK_MODE == "off" or not PK.supported(sh, mode, T, T):
        return False
    a_pk, _ = PK.pack_act(a, None, T, phase_split=(mode == 0 and sh.stride_h == 2))
    w_img = PK.pack_weight(sh, mode, T, T, w_f32=w)
    rc = _timed("fwd_pk" if mode == 0 else "dgrad_pk", sh, lambda: PK.conv(sh, mode, a_pk, T, w_img, T, out))
    if rc == L.E_UNSUPPORTED:
        return False
    L.check(rc, "pk_conv (plain)")
    return True


class ConvTranspose2dFn(Function):
    """y = F.conv_transpose2d(x, w, bias, stride, padding, output_padding, groups, dilation) on the engine's convolution
    kernels.  A transposed convolution IS the data gradient of the convolution S that maps y-space to x-space (w is
    already stored as S's weight [K = C_in][C_out / g][R][S]):

        forward   y  = dgrad_S(dy := x, w)            backward  dx = fwd_S(gy, w),  dw = wgrad_S(x := gy, dy := x)

    so the three kernels of QuantConv2dFn serve it with the roles swapped: the packed-operand tensor-core family where it
    has cover (exact bf16 pieces of the fp32 operands), the generic implicit-GEMM kernels elsewhere."""

    @staticmethod
    def forward(ctx, x, w, bias, stride, padding, output_padding, groups, dilation):
        L.require_cuda(x, w)
        L.require_f32(x, w)
        lib = L.load()
        x, w = x.contiguous(), w.contiguous()
        b, cin, h, wd = x.shape
        if w.shape[0] != cin or cin % groups:
            raise ValueError("conv_transpose2d: weight must be [C_in, C_out / groups, R, S]")
        cout = w.shape[1] * groups
        oh = (h - 1) * stride[0] - 2 * padding[0] + dilation[0] * (w.shape[2] - 1) + output_padding[0] + 1
        ow = (wd - 1) * stride[1] - 2 * padding[1] + dilation[1] * (w.shape[3] - 1) + output_padding[1] + 1
        sh = _shape_struct((b, cout, oh, ow), w.shape, stride, padding, dilation, groups)
        if _out_hw(sh) != (h, wd):
            raise ValueError("conv_transpose2d: output_padding must be smaller than the stride")
        y = torch.empty((b, cout, oh, ow), dtype=torch.float32, device=x.device)
        if not _pk_plain(sh, 1, x, w, y, L.PK_TERMS):
            L.check(_timed("dgrad", sh, lambda: lib.mnb_conv2d_dgrad(C.byref(sh), x.data_ptr(), w.data_ptr(), None, None,
                                                                      y.data_ptr(), L.stream())), "conv2d_dgrad")
        if bias is not None:
            y += bias.view(1, -1, 1, 1)
        ctx.save_for_backward(x, w)
        ctx.sh, ctx.has_bias = sh, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        from . import pk as PK
        lib = L.load()
        x, w = ctx.saved_tensors
        sh = ctx.sh
        gy = gy.contiguous()
        gx = gw = gb = None
        T = min(L.PK_TERMS, L.PK_TERMS_BWD)
        if ctx.needs_input_grad[0]:
            gx = torch.empty_like(x)
            if not _pk_plain(sh, 0, gy, w, gx, T):
                ops = L.ConvOperands()
                ops.a_f32, ops.w_f32 = gy.data_ptr(), w.data_ptr()
                L.check(_timed("fwd", sh, lambda: lib.mnb_conv2d_fwd(C.byref(sh), C.byref(ops), gx.data_ptr(), L.stream())),
                        "conv2d_fwd")
        if ctx.needs_input_grad[1]:
            gw = torch.empty_like(w)
            done = False
            if L.PK_MODE != "off" and PK.wgrad_supported(sh, T, T):
                x_pk, _ = PK.pack_act(x, None, T)                                   # S's output-gradient operand
                g_pk, _ = PK.pack_act(gy, None, T, phase_split=sh.stride_h == 2)    # S's input operand
                rc = _timed("wgrad_pk", sh, lambda: PK.wgrad(sh, x_pk, T, g_pk, T, gw))
                if rc != L.E_UNSUPPORTED:
                    L.check(rc, "pk_wgrad (transposed conv)")
                    done = True
            if not done:
                ops = L.ConvOperands()
                ops.a_f32 = gy.data_ptr()
                ws = torch.empty(max(int(lib.mnb_wgrad_scratch_bytes(C.byref(sh))), 4), dtype=torch.uint8, device=gy.device)
                L.check(_timed("wgrad", sh, lambda: lib.mnb_conv2d_wgrad(C.byref(sh), x.data_ptr(), C.byref(ops), gw.data_ptr(),
                                                                         ws.data_ptr(), L.stream())), "conv2d_wgrad")
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = channel_sums(gy)
        return gx, gw, gb, None, None, None, None, None


def conv_transpose2d(x, w, bias, stride, padding, output_padding, groups, dilation):
    return ConvTranspose2dFn.apply(x, w, bias, tuple(stride), tuple(padding), tuple(output_padding), groups, tuple(dilation))


# --------------------------------------------------------------------------
# frozen inference graphs (iao.freeze_inference): producer -> consumer hand-off of packed operand planes
# --------------------------------------------------------------------------
class Consumer:
    """the quantized conv that reads a producer's output next (set up by iao.freeze_inference): its frozen activation
    quantizer, the nn.ReLU in between (folded away), its geometry, and whether anybody else needs the fp32 tensor"""

    def __init__(self, module, spec, relu, only, w_shape, stride, padding, dilation, groups, int_weights):
        self.module, self.spec, self.relu, self.only = module, spec, bool(relu), bool(only)
        self.w_shape, self.stride, self.padding, self.dilation, self.groups = w_shape, stride, padding, dilation, groups
        self.int_weights = int_weights

    def accepts(self, act_shape):
        """will the consumer's forward run on the packed-operand family with a one-piece plane of this activation?"""
        from . import pk as PK
        sp = self.spec
        if sp is None or not self.int_weights or not (2 <= sp.bits <= 8) or _pk_terms(sp, True)[0] != 1:
            return False
        if act_shape[1] != self.w_shape[1] * self.groups:
            return False
        sh = _shape_struct(act_shape, self.w_shape, self.stride, self.padding, self.dilation, self.groups)
        if sh.stride_h == 2 and ((act_shape[2] | act_shape[3]) & 1):
            return False
        return L.PK_MODE != "off" and PK.supported(sh, 0, 1, 1)

    @property
    def split(self):
        return self.stride[0] == 2


def handed_plane(module, x):
    """the operand plane a producer wrote for ``module`` (None if ``x`` does not carry one that is still valid)"""
    pre = getattr(x, "_mnb_pk_pre", None)
    if pre is not None and pre[0] is module and (x.device.type == "meta" or x._version == pre[2]):
        return pre[1]
    if x.device.type == "meta":
        raise RuntimeError("micronet_b200: a plane-only producer output reached a module it was not produced for")
    return None


def _tag(y, consumer, plane):
    y._mnb_pk_pre = (consumer.module, plane, y._version)
    return y


@torch.no_grad()
def frozen_conv(x, plane, wq, bias, w_int, w_scale, spec, stride, padding, dilation, groups, pre_relu=False, consumer=None):
    """eval forward of a frozen quantized conv.  ``plane``: operand plane its producer already wrote (x holds no data
    then); ``consumer``: write the next conv's plane from the epilogue (mnb_pk_conv_post)."""
    from . import pk as PK
    stride, padding, dilation = tuple(stride), tuple(padding), tuple(dilation)
    sh = _shape_struct(x.shape, wq.shape, stride, padding, dilation, groups)
    p, q = _out_hw(sh)
    out_shape = (x.shape[0], wq.shape[0], p, q)
    fused = consumer is not None and consumer.accepts(out_shape)
    ta, tw = _pk_terms(spec, w_int)
    if (plane is None and not fused) or spec is None or w_int is None or L.PK_MODE == "off" or not PK.supported(sh, 0, ta, tw):
        if plane is not None:
            raise RuntimeError("micronet_b200: handed-over plane in front of a conv outside the packed-operand cover")
        return quant_conv2d(x, wq, bias, w_int, w_scale, spec, stride, padding, dilation, groups, pre_relu=pre_relu)
    dev = wq.device
    if plane is None:
        L.require_cuda(x, wq)
        plane, _ = PK.pack_act(x.contiguous(), spec.struct(), ta, phase_split=sh.stride_h == 2, relu=pre_relu)
    cache = getattr(w_int, "_mnb_pk_cache", None)
    ckey = (PK._key(sh), ta, tw)
    w_img = cache.get(ckey) if cache is not None else None
    if w_img is None:
        w_img = PK.pack_weight(sh, 0, ta, tw, w_int=w_int)
        if cache is not None:
            cache[ckey] = w_img
    a_scale = spec.scale if spec.mode == L.ACT_IAO else None
    a_const = 1.0 / float(2 ** spec.bits - 1) if spec.mode == L.ACT_DOREFA else 1.0
    if not fused:
        y = torch.empty(out_shape, dtype=torch.float32, device=dev)
        L.check(_timed("fwd_pk", sh, lambda: PK.conv(sh, 0, plane, ta, w_img, tw, y, n_scale=w_scale, a_scale=a_scale,
                                                     a_scale_const=a_const, bias=bias)), "pk_conv fwd")
        return y
    y = None if consumer.only else torch.empty(out_shape, dtype=torch.float32, device=dev)
    cplane = PK.consumer_plane(*out_shape, dev)
    cqp = consumer.spec.struct()
    L.check(_timed("fwd_pk", sh, lambda: PK.conv_post(sh, plane, ta, w_img, tw, y, cqp, cplane, consumer.relu, consumer.split,
                                                      n_scale=w_scale, a_scale=a_scale, a_scale_const=a_const, bias=bias)),
            "pk_conv_post")
    if y is None:
        y = torch.empty(out_shape, dtype=torch.float32, device="meta")   # shape only: the data lives in the consumer's plane
    return _tag(y, consumer, cplane)


@torch.no_grad()
def frozen_quant_add(a, b, spec, relu, consumer=None):
    """eval forward of a frozen QuantAdd; with a ``consumer`` the kernel also writes the next conv's operand plane"""
    if consumer is None or not consumer.accepts(tuple(a.shape)) or a.dim() != 4:
        return QuantAddFn.apply(a, b, spec, relu)
    from . import pk as PK
    L.require_cuda(a, b)
    lib = L.load()
    a, b = a.contiguous(), b.contiguous()
    assert a.shape == b.shape, "QuantAdd: operand shapes differ"
    out = torch.empty_like(a)
    cplane = PK.consumer_plane(*a.shape, a.device)
    qp, cqp = spec.struct(), consumer.spec.struct()
    post = L.PkPost(C.pointer(cqp), 1 if (consumer.relu and not relu) else 0, 1 if consumer.split else 0, cplane.data_ptr())
    L.check(lib.mnb_quant_add_pack_fwd(a.data_ptr(), b.data_ptr(), a.shape[0], a.shape[1], a.shape[2], a.shape[3],
                                       C.byref(qp), 1 if relu else 0, out.data_ptr(), C.byref(post), L.stream()),
            "quant_add_pack_fwd")
    return _tag(out, consumer, cplane)


def quant_linear(x, wq, bias, w_int, w_scale, spec):
    """F.linear on the same kernels: [*, C] -> 1x1 conv on a [N, C, 1, 1] view."""
    lead = x.shape[:-1]
    x4 = x.reshape(-1, x.shape[-1], 1, 1)
    w4 = wq.reshape(wq.shape[0], wq.shape[1], 1, 1)
    wi4 = None if w_int is None else w_int.reshape(w4.shape)
    y = QuantConv2dFn.apply(x4, w4, bias, wi4, w_scale, spec, (1, 1), (0, 0), (1, 1), 1)
    return y.reshape(*lead, wq.shape[0])


class BNFoldFn(Function):
    """IAO:903-945: (weight, bias) with the BatchNorm statistics folded in, one kernel each way"""

    @staticmethod
    def forward(ctx, weight, bias, gamma, beta, mean, var, eps):
        L.require_cuda(weight, gamma)
        lib = L.load()
        weight = weight.contiguous()
        k, n = weight.shape[0], weight.numel() // weight.shape[0]
        mean, var = mean.contiguous(), var.contiguous()
        w_f = torch.empty_like(weight)
        b_f = torch.empty(k, dtype=torch.float32, device=weight.device)
        L.check(lib.mnb_bn_fold_fwd(weight.data_ptr(), k, n, gamma.data_ptr(), beta.data_ptr(), L.ptr(bias), mean.data_ptr(),
                                    var.data_ptr(), float(eps), w_f.data_ptr(), b_f.data_ptr(), L.stream()), "bn_fold_fwd")
        ctx.save_for_backward(weight, bias, gamma, mean, var)
        ctx.eps = eps
        return w_f, b_f

    @staticmethod
    def backward(ctx, dw_f, db_f):
        lib = L.load()
        weight, bias, gamma, mean, var = ctx.saved_tensors
        k, n = weight.shape[0], weight.numel() // weight.shape[0]
        if dw_f is None:
            dw_f = torch.zeros_like(weight)
        dw_f = dw_f.contiguous()
        db_f = None if db_f is None else db_f.contiguous()
        dw = torch.empty_like(weight) if ctx.needs_input_grad[0] else None
        out6 = torch.empty((k, 6), dtype=torch.float32, device=weight.device)
        L.check(lib.mnb_bn_fold_bwd(dw_f.data_ptr(), L.ptr(db_f), weight.data_ptr(), k, n, gamma.data_ptr(), L.ptr(bias),
                                    mean.data_ptr(), var.data_ptr(), float(ctx.eps), L.ptr(dw), out6.data_ptr(), L.stream()),
                "bn_fold_bwd")
        g = ctx.needs_input_grad
        return (dw, out6[:, 2] if (bias is not None and g[1]) else None, out6[:, 0] if g[2] else None,
                out6[:, 1] if g[3] else None, out6[:, 3] if g[4] else None, out6[:, 4] if g[5] else None, None)


# --------------------------------------------------------------------------
# per-channel batch statistics (BN-fuse training path, IAO:853-855)
# --------------------------------------------------------------------------
class ChannelMeanVarFn(Function):
    @staticmethod
    def forward(ctx, x):
        L.require_cuda(x)
        lib = L.load()
        x = x.contiguous()
        b, c = x.shape[0], x.shape[1]
        hw = x.numel() // (b * c)
        out = torch.empty(2 * c, dtype=torch.float32, device=x.device)
        L.check(lib.mnb_channel_stats(x.data_ptr(), b, c, hw, 1, out.data_ptr(),
                                      L.scratch(x.device, c).data_ptr(), L.stream()), "channel_stats")
        mean, var = out[:c], out[c:]
        ctx.save_for_backward(x, mean)
        return mean, var

    @staticmethod
    def backward(ctx, dmean, dvar):
        lib = L.load()
        x, mean = ctx.saved_tensors
        b, c = x.shape[0], x.shape[1]
        hw = x.numel() // (b * c)
        dmean = torch.zeros_like(mean) if dmean is None else dmean.contiguous()
        dvar = torch.zeros_like(mean) if dvar is None else dvar.contiguous()
        dx = torch.empty_like(x)
        L.check(lib.mnb_channel_stats_bwd(x.data_ptr(), mean.contiguous().data_ptr(), dmean.data_ptr(),
                                          dvar.data_ptr(), b, c, hw, dx.data_ptr(), L.stream()),
                "channel_stats_bwd")
        return dx


def channel_mean_var(x):
    return ChannelMeanVarFn.apply(x)
