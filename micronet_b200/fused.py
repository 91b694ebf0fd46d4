"""Producer-side fusion (SURVEY.md 8 f2) for wbwtab-prepared models.

A wbwtab block is ``[channel_shuffle ->] conv -> bn -> ActivationQuantizer(A=2)`` (nin_gc.py:36-59 with the
ReLU swapped by WB:319-322), optionally followed by ``nn.MaxPool2d``.  ``fuse_wbwtab_blocks`` rewrites, in place:

* every sibling pair (BatchNorm2d, ActivationQuantizer(A=2)) -> (``BatchNormBinarize2d``, Identity): batch
  statistics, normalise + sign + STE mask in two kernels forward and two backward; the backward also hands the
  producing convolution its bias gradient (channel sums of dx), saving that pass;
* every plain ``nn.MaxPool2d`` -> ``EngineMaxPool2d`` (byte window index, bit-identical to ATen); a 2x2 pool
  that directly follows a fused BN+binarizer is absorbed by it (the un-pooled +-1 tensor is never written);
* the un-quantized first ``nn.Conv2d`` (few input channels) -> ``EngineFloatConv2d``: fp32-accurate im2col
  convolution on the tensor cores (forward + weight gradient);
* every block whose input shuffle (``channel_shuffle_flag`` / ``shuffle_groups`` attributes of the
  reference's block class) directly follows one of those producers: the permutation moves into the producer's
  output addressing and the shuffle copy disappears (max-pooling commutes with a channel permutation).

Parameters, buffers, state_dict keys and the numbers are unchanged; only intermediate tensors between a
producer and a shuffled block are stored in the shuffled channel order."""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.autograd import Function

import ctypes as C

import torch.nn.functional as TF

from . import _lib as L


class BNSignFn(Function):
    """sign(batch_norm(x)) [-> max_pool2d(2, 2)] [-> channel_shuffle] with the saturate STE"""

    @staticmethod
    def forward(ctx, x, gamma, beta, mean, invstd, training, shuffle_groups, pool, plane_only=False):
        lib = L.load()
        x = x.contiguous()
        b, c = x.shape[0], x.shape[1]
        hw = x.numel() // (b * c)
        bits = torch.empty((x.numel() + 31) // 32, dtype=torch.int32, device=x.device)
        arg = None
        if pool:
            h, w = x.shape[2], x.shape[3]
            y = torch.empty((b, c, h // 2, w // 2), dtype=x.dtype, device=x.device)
            arg = torch.empty(y.numel(), dtype=torch.uint8, device=x.device)
            L.check(lib.mnb_bn_sign_pool_fwd(x.data_ptr(), b, c, h, w, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                             beta.data_ptr(), shuffle_groups, y.data_ptr(), bits.data_ptr(), arg.data_ptr(),
                                             L.stream()), "bn_sign_pool_fwd")
        else:
            y = torch.empty_like(x)
            rc = L.E_UNSUPPORTED
            if c % 8 == 0 and hw % 32 == 0 and x.dim() == 4 and L.PK_MODE != "off":
                # the +-1 output also as the operand plane of the consuming conv (packed-operand family): 2 extra bytes per
                # element here save that conv's 4-byte read and its pack pass
                plane = torch.empty(x.numel() * 2, dtype=torch.uint8, device=x.device)
                # plane_only (set by the rewrite pass when the ONLY reader is a conv of the packed-operand family): the fp32
                # tensor is a shape-carrying placeholder, 4 of the 10 bytes per element this pass moved are never written
                skip_y = bool(plane_only) and L.PLANE_ONLY
                rc = lib.mnb_bn_sign_fwd_packed(x.data_ptr(), b, c, hw, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                                beta.data_ptr(), shuffle_groups, None if skip_y else y.data_ptr(),
                                                bits.data_ptr(), plane.data_ptr(), L.stream())
                if rc == 0:
                    y._mnb_pk_pm1 = plane
                    if skip_y:
                        y._mnb_plane_only = True    # functional.materialized(y) rebuilds the values from the plane
                elif rc != L.E_UNSUPPORTED:
                    L.check(rc, "bn_sign_fwd_packed")
            if rc != 0:
                L.check(lib.mnb_bn_sign_fwd(x.data_ptr(), b, c, hw, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                            beta.data_ptr(), shuffle_groups, y.data_ptr(), bits.data_ptr(), L.stream()),
                        "bn_sign_fwd")
        y._mnb_pm1 = True        # exactly +-1: a consuming conv may pack it as ONE bf16 piece
        ctx.save_for_backward(x, gamma, mean, invstd)
        ctx.bits, ctx.arg, ctx.training, ctx.shuffle_groups = bits, arg, training, shuffle_groups
        # the conv that produced x ran on the packed-operand family (functional.QuantConv2dFn tags its output): its
        # gradient operand is written by this backward, pre-multiplied with the conv's per-channel weight scale
        ctx.pk_conv = getattr(x, "_mnb_pk_conv", None)
        return y

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        x, gamma, mean, invstd = ctx.saved_tensors
        g = g.contiguous()
        b, c = x.shape[0], x.shape[1]
        hw = x.numel() // (b * c)
        dx = torch.empty_like(x)
        out = torch.empty(3 * c, dtype=torch.float32, device=x.device)
        dgamma, dbeta, dx_sum = out[:c], out[c:2 * c], out[2 * c:]
        scratch = L.scratch(x.device, c)
        if (ctx.arg is not None and ctx.pk_conv is not None and ctx.training and c % 8 == 0 and x.shape[3] % 8 == 0
                and x.shape[2] % 2 == 0):
            # pooled producer behind a conv of the packed-operand family: reduce pass (dgamma, dbeta), then the apply pass
            # writes the full-resolution gradient straight as that conv's packed operand (no fp32 dx, no pack pass)
            w_scale, T = ctx.pk_conv
            L.check(lib.mnb_bn_sign_pool_bwd(g.data_ptr(), ctx.bits.data_ptr(), ctx.arg.data_ptr(), x.data_ptr(), b, c,
                                             x.shape[2], x.shape[3], mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                             2, ctx.shuffle_groups, dx.data_ptr(), dgamma.data_ptr(),
                                             dbeta.data_ptr(), None, scratch.data_ptr(), L.stream()), "bn_sign_pool_bwd (reduce)")
            dy_pk = torch.empty(T * x.numel() * 2, dtype=torch.uint8, device=x.device)
            L.check(lib.mnb_bn_sign_pool_bwd_pack(g.data_ptr(), ctx.bits.data_ptr(), ctx.arg.data_ptr(), x.data_ptr(), b, c,
                                                  x.shape[2], x.shape[3], mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                                  dgamma.data_ptr(), dbeta.data_ptr(), ctx.shuffle_groups, L.ptr(w_scale), T,
                                                  dy_pk.data_ptr(), L.stream()), "bn_sign_pool_bwd_pack")
            dx_sum.zero_()
            dx._mnb_pk_dy = (dy_pk, T, w_scale)     # dx itself is NOT written: its only reader is that conv's backward
        elif ctx.arg is not None:
            L.check(lib.mnb_bn_sign_pool_bwd(g.data_ptr(), ctx.bits.data_ptr(), ctx.arg.data_ptr(), x.data_ptr(), b, c,
                                             x.shape[2], x.shape[3], mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                             1 if ctx.training else 0, ctx.shuffle_groups, dx.data_ptr(), dgamma.data_ptr(),
                                             dbeta.data_ptr(), dx_sum.data_ptr(), scratch.data_ptr(), L.stream()),
                    "bn_sign_pool_bwd")
        elif ctx.pk_conv is not None and ctx.training and c % 8 == 0:
            # reduce pass of mnb_bn_sign_bwd (dgamma, dbeta), then the apply pass that writes dx as the producing conv's packed
            # gradient operand.  The channel sums of dx (that conv's bias gradient) are exactly zero behind a training-mode
            # BatchNorm; the reference's value is the rounding noise of that sum.
            w_scale, T = ctx.pk_conv
            L.check(lib.mnb_bn_sign_bwd(g.data_ptr(), ctx.bits.data_ptr(), x.data_ptr(), b, c, hw, mean.data_ptr(),
                                        invstd.data_ptr(), gamma.data_ptr(), 2, ctx.shuffle_groups,
                                        dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), None,
                                        scratch.data_ptr(), L.stream()), "bn_sign_bwd (reduce)")
            dy_pk = torch.empty(T * x.numel() * 2, dtype=torch.uint8, device=x.device)
            L.check(lib.mnb_bn_sign_bwd_pack(g.data_ptr(), ctx.bits.data_ptr(), x.data_ptr(), b, c, hw, mean.data_ptr(),
                                             invstd.data_ptr(), gamma.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(),
                                             ctx.shuffle_groups, L.ptr(w_scale), T, None, dy_pk.data_ptr(), L.stream()),
                    "bn_sign_bwd_pack")
            dx_sum.zero_()
            dx._mnb_pk_dy = (dy_pk, T, w_scale)     # dx itself is NOT written: its only reader is that conv's backward
        else:
            L.check(lib.mnb_bn_sign_bwd(g.data_ptr(), ctx.bits.data_ptr(), x.data_ptr(), b, c, hw, mean.data_ptr(),
                                        invstd.data_ptr(), gamma.data_ptr(), 1 if ctx.training else 0, ctx.shuffle_groups,
                                        dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), dx_sum.data_ptr(),
                                        scratch.data_ptr(), L.stream()), "bn_sign_bwd")
        # picked up by QuantConv2dFn.backward when this dx is its grad_output (saves its own channel-sum pass)
        dx._mnb_channel_sum = dx_sum
        return dx, dgamma, dbeta, None, None, None, None, None, None


class BatchNormBinarize2d(nn.BatchNorm2d):
    """nn.BatchNorm2d followed by wbwtab's binarizing ActivationQuantizer.  ``pool2`` additionally applies the
    nn.MaxPool2d(2, 2) that follows the block; ``out_shuffle_groups`` > 1 writes the result in the channel
    order ``shuffle_channels(., groups)`` would produce."""

    out_shuffle_groups = 1
    pool2 = False
    plane_only = False     # set by fuse_wbwtab_blocks: the only reader of the output is a conv that takes the bf16 plane

    def forward(self, input):
        L.require_cuda(input, self.weight)
        L.require_f32(input, self.weight)
        assert self.affine and self.track_running_stats and self.momentum is not None, \
            "BatchNormBinarize2d supports affine BN with running statistics and a float momentum"
        if self.training:
            lib = L.load()
            x = input.detach().contiguous()
            b, c = x.shape[0], x.shape[1]
            stats = torch.empty(2 * c, dtype=torch.float32, device=x.device)
            L.check(lib.mnb_bn_batch_stats(x.data_ptr(), b, c, x.numel() // (b * c), float(self.eps), float(self.momentum),
                                           self.running_mean.data_ptr(), self.running_var.data_ptr(),
                                           self.num_batches_tracked.data_ptr(), stats.data_ptr(),
                                           L.scratch(x.device, c).data_ptr(), L.stream()), "bn_batch_stats")
            mean, invstd = stats[:c], stats[c:]
        else:
            mean = self.running_mean
            invstd = torch.rsqrt(self.running_var + self.eps)
        sg = int(self.out_shuffle_groups)
        if self.pool2 and (input.dim() != 4 or input.shape[2] % 2 or input.shape[3] % 8):
            # plane shape outside the fused pool kernel's cover: the same result in two steps
            y = BNSignFn.apply(input, self.weight, self.bias, mean, invstd, self.training, 1, False)
            return MaxPoolFn.apply(y, 2, 2, 0, sg)
        return BNSignFn.apply(input, self.weight, self.bias, mean, invstd, self.training, sg, bool(self.pool2),
                              bool(self.plane_only) and not self.pool2)

    def extra_repr(self):
        return super().extra_repr() + f", pool2={self.pool2}, out_shuffle_groups={self.out_shuffle_groups}"



class BNReluQuantFn(Function):
    """BatchNorm2d -> ReLU -> DoReFa activation quantizer of the NEXT conv, written as that conv's packed bf16 operand.
    The returned fp32 tensor is a shape-carrying placeholder (never written, never read): its only consumer is the
    engine QuantConv2d the rewrite pass found behind this block, which reads ``_mnb_pk_q`` instead."""

    @staticmethod
    def forward(ctx, x, gamma, beta, mean, invstd, training, shuffle_groups, a_bits):
        from . import functional as F_
        lib = L.load()
        x = x.contiguous()
        b, c = x.shape[0], x.shape[1]
        hw = x.numel() // (b * c)
        bits = torch.empty((x.numel() + 31) // 32, dtype=torch.int32, device=x.device)
        packed = torch.empty(x.numel() * 2, dtype=torch.uint8, device=x.device)
        qp = F_.ActSpec(L.ACT_DOREFA, bits=a_bits).struct()
        L.check(lib.mnb_bn_relu_quant_pack_fwd(x.data_ptr(), b, c, hw, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                               beta.data_ptr(), C.byref(qp), shuffle_groups, packed.data_ptr(),
                                               bits.data_ptr(), L.stream()), "bn_relu_quant_pack_fwd")
        y = torch.empty_like(x)                      # placeholder: allocation only, no kernel
        y._mnb_pk_q = (packed, a_bits)               # picked up by QuantConv2dFn.forward
        ctx.save_for_backward(x, gamma, mean, invstd)
        ctx.bits, ctx.training, ctx.shuffle_groups = bits, training, shuffle_groups
        return y

    @staticmethod
    def backward(ctx, g):
        # g = d loss / d (quantized conv input) already multiplied by the quantizer's 0.1 (the conv's data-gradient epilogue);
        # the combined mask relu'(bn) * [0.1 bn <= 1] and the BatchNorm backward are mnb_bn_sign_bwd's job
        lib = L.load()
        x, gamma, mean, invstd = ctx.saved_tensors
        g = g.contiguous()
        b, c = x.shape[0], x.shape[1]
        hw = x.numel() // (b * c)
        dx = torch.empty_like(x)
        out = torch.empty(3 * c, dtype=torch.float32, device=x.device)
        dgamma, dbeta, dx_sum = out[:c], out[c:2 * c], out[2 * c:]
        L.check(lib.mnb_bn_sign_bwd(g.data_ptr(), ctx.bits.data_ptr(), x.data_ptr(), b, c, hw, mean.data_ptr(),
                                    invstd.data_ptr(), gamma.data_ptr(), 1 if ctx.training else 0, ctx.shuffle_groups,
                                    dx.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), dx_sum.data_ptr(),
                                    L.scratch(x.device, c).data_ptr(), L.stream()), "bn_sign_bwd")
        dx._mnb_channel_sum = dx_sum
        return dx, dgamma, dbeta, None, None, None, None, None


class BatchNormReluQuant2d(nn.BatchNorm2d):
    """nn.BatchNorm2d + nn.ReLU + the DoReFa activation quantizer (``a_bits``) of the QuantConv2d that consumes this block's
    output, in one pass (SURVEY.md 8 f2).  Parameters, buffers and state_dict keys are those of the BatchNorm2d it replaces;
    ``out_shuffle_groups`` as in BatchNormBinarize2d.  Planes outside the fused kernel's cover (C % 8, H*W % 32) fall back
    to the un-fused sequence."""

    out_shuffle_groups = 1
    a_bits = 8

    def forward(self, input):
        L.require_cuda(input, self.weight)
        L.require_f32(input, self.weight)
        b, c = input.shape[0], input.shape[1]
        hw = input.numel() // max(1, b * c)
        sg = int(self.out_shuffle_groups)
        if input.dim() != 4 or c % 8 or hw % 32:
            y = TF.relu(super().forward(input))
            if sg > 1:
                y = y.view(b, sg, c // sg, *y.shape[2:]).transpose(1, 2).contiguous().view_as(y)
            return y
        if self.training:
            lib = L.load()
            x = input.detach().contiguous()
            stats = torch.empty(2 * c, dtype=torch.float32, device=x.device)
            L.check(lib.mnb_bn_batch_stats(x.data_ptr(), b, c, hw, float(self.eps), float(self.momentum),
                                           self.running_mean.data_ptr(), self.running_var.data_ptr(),
                                           self.num_batches_tracked.data_ptr(), stats.data_ptr(),
                                           L.scratch(x.device, c).data_ptr(), L.stream()), "bn_batch_stats")
            mean, invstd = stats[:c], stats[c:]
        else:
            mean = self.running_mean
            invstd = torch.rsqrt(self.running_var + self.eps)
        return BNReluQuantFn.apply(input, self.weight, self.bias, mean, invstd, self.training, sg, int(self.a_bits))

    def extra_repr(self):
        return super().extra_repr() + f", relu + dorefa a_bits={self.a_bits}, out_shuffle_groups={self.out_shuffle_groups}"


class MaxPoolFn(Function):
    @staticmethod
    def forward(ctx, x, k, s, p, shuffle_groups):
        lib = L.load()
        x = x.contiguous()
        b, c, h, w = x.shape
        oh, ow = (h + 2 * p - k) // s + 1, (w + 2 * p - k) // s + 1
        y = torch.empty((b, c, oh, ow), dtype=x.dtype, device=x.device)
        arg = torch.empty(y.numel(), dtype=torch.uint8, device=x.device)
        L.check(lib.mnb_maxpool2d_fwd(x.data_ptr(), b, c, h, w, k, s, p, shuffle_groups, y.data_ptr(), arg.data_ptr(),
                                      L.stream()), "maxpool2d_fwd")
        ctx.arg, ctx.cfg = arg, (b, c, h, w, k, s, p, shuffle_groups)
        return y

    @staticmethod
    def backward(ctx, g):
        lib = L.load()
        b, c, h, w, k, s, p, sg = ctx.cfg
        g = g.contiguous()
        dx = torch.empty((b, c, h, w), dtype=g.dtype, device=g.device)
        L.check(lib.mnb_maxpool2d_bwd(g.data_ptr(), ctx.arg.data_ptr(), b, c, h, w, k, s, p, sg, dx.data_ptr(),
                                      L.stream()), "maxpool2d_bwd")
        return dx, None, None, None, None


def _pool_cfg(m: nn.MaxPool2d):
    """(k, s, p) if the engine kernel covers this pool (square, dilation 1, floor mode), else None"""
    def one(v):
        if isinstance(v, (tuple, list)):
            return int(v[0]) if len(set(v)) == 1 else None
        return int(v)
    k, s, p, d = one(m.kernel_size), one(m.stride if m.stride is not None else m.kernel_size), one(m.padding), one(m.dilation)
    if None in (k, s, p, d) or d != 1 or m.ceil_mode or m.return_indices or k > 15 or 2 * p > k:
        return None
    return k, s, p


class EngineMaxPool2d(nn.MaxPool2d):
    out_shuffle_groups = 1

    def forward(self, input):
        L.require_cuda(input)
        L.require_f32(input)
        k, s, p = _pool_cfg(self)
        return MaxPoolFn.apply(input, k, s, p, int(self.out_shuffle_groups))

    def extra_repr(self):
        return super().extra_repr() + f", out_shuffle_groups={self.out_shuffle_groups}"


class FloatConvFn(Function):
    """fp32 conv2d with few input channels on the tensor-core im2col path (mnb_fconv2d_*_tc);
    shapes outside its cover run ATen's convolution (what the reference runs for this layer)."""

    @staticmethod
    def forward(ctx, x, w, bias, padding):
        lib = L.load()
        x, w = x.contiguous(), w.contiguous()
        b, c, h, wd = x.shape
        k, _, r, s_ = w.shape
        sh = L.ConvShape(b, c, h, wd, k, r, s_, 1, 1, padding, padding, 1, 1, 1)
        y = torch.empty((b, k, h, wd), dtype=torch.float32, device=x.device)
        rc = lib.mnb_fconv2d_fwd_tc(C.byref(sh), x.data_ptr(), w.data_ptr(), L.ptr(bias), y.data_ptr(),
                                    L.tc_err_flag(x.device).data_ptr(), L.stream())
        ctx.engine = rc == 0
        if rc == L.E_UNSUPPORTED:
            y = TF.conv2d(x, w, bias, 1, padding)
        elif rc != 0:
            L.check(rc, "fconv2d_fwd_tc")
        ctx.save_for_backward(x, w)
        ctx.sh, ctx.padding, ctx.has_bias = sh, padding, bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        x, w = ctx.saved_tensors
        presummed = getattr(dy, "_mnb_channel_sum", None)
        dy = dy.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.nn.grad.conv2d_input(x.shape, w, dy, 1, ctx.padding)
        if ctx.needs_input_grad[1]:
            need = int(lib.mnb_fconv2d_wgrad_tc_scratch_bytes(C.byref(ctx.sh))) if ctx.engine else -1
            if need >= 0:
                dw = torch.empty_like(w)
                scratch = torch.empty(need, dtype=torch.uint8, device=dy.device)
                L.check(lib.mnb_fconv2d_wgrad_tc(C.byref(ctx.sh), dy.data_ptr(), x.data_ptr(), dw.data_ptr(),
                                                 scratch.data_ptr(), L.tc_err_flag(dy.device).data_ptr(), L.stream()),
                        "fconv2d_wgrad_tc")
            else:
                dw = torch.nn.grad.conv2d_weight(x, w.shape, dy, 1, ctx.padding)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            if presummed is not None and presummed.numel() == dy.shape[1]:
                db = presummed
            else:
                from .functional import channel_sums
                db = channel_sums(dy)
        return dx, dw, db, None


def _float_conv_cover(m: nn.Conv2d) -> bool:
    k, p = m.kernel_size, m.padding
    return (type(m) is nn.Conv2d and m.groups == 1 and tuple(m.stride) == (1, 1) and tuple(m.dilation) == (1, 1)
            and k[0] == k[1] and k[0] % 2 == 1 and not isinstance(p, str) and tuple(p) == (k[0] // 2, k[0] // 2)
            and m.padding_mode == "zeros" and m.in_channels * k[0] * k[1] <= 128 and m.out_channels <= 256)


class EngineFloatConv2d(nn.Conv2d):
    """drop-in for the un-quantized first nn.Conv2d of a QAT model (same parameters / state_dict keys)"""

    def forward(self, input):
        L.require_cuda(input, self.weight)
        L.require_f32(input, self.weight)
        return FloatConvFn.apply(input, self.weight, self.bias, int(self.padding[0]))


class EnginePmConv2d(nn.Conv2d):
    """drop-in for an un-quantized nn.Conv2d that reads a binarizer's +-1 output (wbwtab leaves the last conv of a model in
    fp32, WB:247-331): on the packed-operand tensor-core family when its input carries the +-1 tag and the shape is inside
    the family's cover (forward and both gradients), otherwise exactly the stock convolution.  Same parameters / state_dict."""

    def forward(self, input):
        from . import functional as F_, pk as PK
        if (getattr(input, "_mnb_pm1", False) and L.PK_MODE != "off" and input.is_cuda and input.dtype == torch.float32
                and input.dim() == 4 and self.padding_mode == "zeros" and not isinstance(self.padding, str)):
            sh = F_._shape_struct(input.shape, self.weight.shape, self.stride, self.padding, self.dilation, self.groups)
            T, Tb = L.PK_TERMS, min(L.PK_TERMS, L.PK_TERMS_BWD)
            if (PK.supported(sh, 0, 1, T) and PK.supported(sh, 1, Tb, Tb) and PK.wgrad_supported(sh, Tb, 1)):
                return F_.quant_conv2d(input, self.weight, self.bias, None, None, None, self.stride, self.padding,
                                       self.dilation, self.groups)
        from . import functional as F2
        return self._conv_forward(F2.materialized(input), self.weight, self.bias)


def _fuse_pairs(module: nn.Module):
    from .wbwtab import ActivationQuantizer
    prev_name, prev = None, None
    for name, child in list(module.named_children()):
        if (isinstance(child, ActivationQuantizer) and child.A == 2 and type(prev) is nn.BatchNorm2d
                and prev.affine and prev.track_running_stats and prev.momentum is not None):
            fused = BatchNormBinarize2d(prev.num_features, eps=prev.eps, momentum=prev.momentum)
            fused.weight, fused.bias = prev.weight, prev.bias
            fused.running_mean, fused.running_var = prev.running_mean, prev.running_var
            fused.num_batches_tracked = prev.num_batches_tracked
            fused.train(prev.training)
            module._modules[prev_name] = fused
            module._modules[name] = nn.Identity()
        elif type(child) is nn.Conv2d and _float_conv_cover(child):
            conv = EngineFloatConv2d(child.in_channels, child.out_channels, child.kernel_size, child.stride, child.padding,
                                     child.dilation, child.groups, child.bias is not None)
            conv.weight, conv.bias = child.weight, child.bias
            module._modules[name] = conv
        elif type(child) is nn.Conv2d and child.in_channels % 8 == 0 and child.in_channels >= 64:
            conv = EnginePmConv2d(child.in_channels, child.out_channels, child.kernel_size, child.stride, child.padding,
                                  child.dilation, child.groups, child.bias is not None, child.padding_mode)
            conv.weight, conv.bias = child.weight, child.bias
            module._modules[name] = conv
        elif type(child) is nn.MaxPool2d and _pool_cfg(child) is not None:
            pool = EngineMaxPool2d(child.kernel_size, child.stride, child.padding, child.dilation,
                                   child.return_indices, child.ceil_mode)
            module._modules[name] = pool
        else:
            _fuse_pairs(child)
        prev_name, prev = name, module._modules[name]


def _tail_producer(m: nn.Module):
    """the module whose output IS ``m``'s output, if it is one of the shuffling producers"""
    if isinstance(m, (BatchNormBinarize2d, BatchNormReluQuant2d, EngineMaxPool2d)):
        return m
    if hasattr(m, "channel_shuffle_flag"):  # the reference's conv-bn-act block: children run in order
        kids = [k for k in m.children() if not isinstance(k, nn.Identity)]
        if kids and isinstance(kids[-1], (BatchNormBinarize2d, BatchNormReluQuant2d)):
            return kids[-1]
    return None


def _fold_pools(module: nn.Module):
    """BatchNormBinarize2d directly followed by a 2x2 / stride 2 max-pool sibling -> one fused producer"""
    for child in module.children():
        _fold_pools(child)
    if not isinstance(module, nn.Sequential):
        return
    names = [n for n, k in module.named_children() if not isinstance(k, nn.Identity)]
    for pn, cn in zip(names, names[1:]):
        prev, cur = module._modules[pn], module._modules[cn]
        if not isinstance(cur, EngineMaxPool2d) or _pool_cfg(cur) != (2, 2, 0) or cur.out_shuffle_groups != 1:
            continue
        prod = _tail_producer(prev)
        if isinstance(prod, BatchNormBinarize2d) and not prod.pool2 and prod.out_shuffle_groups == 1:
            prod.pool2 = True
            module._modules[cn] = nn.Identity()


def _fold_shuffles(module: nn.Module):
    for child in module.children():
        _fold_shuffles(child)
    if not isinstance(module, nn.Sequential):
        return
    kids = [k for k in module.children() if not isinstance(k, nn.Identity)]
    for prev, blk in zip(kids, kids[1:]):
        groups = int(getattr(blk, "shuffle_groups", 1))
        if not getattr(blk, "channel_shuffle_flag", 0) or groups <= 1:
            continue
        prod = _tail_producer(prev)
        if prod is None or prod.out_shuffle_groups != 1:
            continue
        prod.out_shuffle_groups = groups
        blk.channel_shuffle_flag = 0


def _first_conv(m: nn.Module):
    """the conv that consumes ``m``'s input first, if ``m`` is a conv or one of the reference's conv-bn-act blocks"""
    if isinstance(m, nn.Conv2d):
        return m
    if hasattr(m, "channel_shuffle_flag"):
        kids = [k for k in m.children() if not isinstance(k, nn.Identity)]
        if kids and isinstance(kids[0], nn.Conv2d):
            return kids[0]
    return None


def _fuse_dorefa_producers(module: nn.Module):
    """conv-bn-relu block directly followed (in an nn.Sequential) by a block whose first conv is a DoReFa QuantConv2d with a
    2..8-bit activation quantizer: BatchNorm2d + ReLU + that quantizer + operand packing become one producer"""
    from .dorefa import QuantConv2d as DorefaConv
    for child in module.children():
        _fuse_dorefa_producers(child)
    if not isinstance(module, nn.Sequential) or "mnb_bn_relu_quant_pack_fwd" not in L.PROTOTYPES:
        return
    kids = [k for k in module.children() if not isinstance(k, nn.Identity)]
    for prev, nxt in zip(kids, kids[1:]):
        conv = _first_conv(nxt)
        a_bits = int(conv.activation_quantizer.a_bits) if isinstance(conv, DorefaConv) else 0
        if not (2 <= a_bits <= 8) or conv.in_channels % 8 or tuple(conv.stride) != (1, 1) or conv.quant_inference:
            continue
        if not hasattr(prev, "channel_shuffle_flag"):
            continue
        names = [n for n, k in prev.named_children() if not isinstance(k, nn.Identity)]
        if len(names) < 2:
            continue
        bn, act = prev._modules[names[-2]], prev._modules[names[-1]]
        if type(bn) is not nn.BatchNorm2d or type(act) is not nn.ReLU:
            continue
        if not (bn.affine and bn.track_running_stats and bn.momentum is not None):
            continue
        fused = BatchNormReluQuant2d(bn.num_features, eps=bn.eps, momentum=bn.momentum)
        fused.weight, fused.bias = bn.weight, bn.bias
        fused.running_mean, fused.running_var = bn.running_mean, bn.running_var
        fused.num_batches_tracked = bn.num_batches_tracked
        fused.a_bits = a_bits
        fused.train(bn.training)
        prev._modules[names[-2]] = fused
        prev._modules[names[-1]] = nn.Identity()


def _mark_plane_only(module: nn.Module):
    """BatchNorm + binarizer whose output is read by exactly one module - the conv that opens the next block of the same
    nn.Sequential, un-shuffled - and that conv is one that takes the producer's bf16 plane (wbwtab QuantConv2d with binary /
    ternary weights, or the +-1-input head EnginePmConv2d): the producer then skips its fp32 output."""
    from .wbwtab import QuantConv2d as WbConv
    for child in module.children():
        _mark_plane_only(child)
    if not isinstance(module, nn.Sequential):
        return
    kids = [k for k in module.children() if not isinstance(k, nn.Identity)]
    for prev, nxt in zip(kids, kids[1:]):
        prod, conv = _tail_producer(prev), _first_conv(nxt)
        if not isinstance(prod, BatchNormBinarize2d) or prod.pool2 or conv is None:
            continue
        if getattr(nxt, "channel_shuffle_flag", 0) or conv.in_channels % 8:
            continue
        if isinstance(conv, WbConv):
            ok = conv.weight_quantizer.W in (2, 3) and not conv.quant_inference
        else:
            ok = isinstance(conv, EnginePmConv2d)
        if ok:
            prod.plane_only = True


def fuse_wbwtab_blocks(model: nn.Module, fold_shuffle: bool = True) -> nn.Module:
    _fuse_pairs(model)
    _fold_pools(model)
    _fuse_dorefa_producers(model)
    if fold_shuffle:
        _fold_shuffles(model)
    _mark_plane_only(model)
    return model


fuse_blocks = fuse_wbwtab_blocks      # the pool / first-conv / shuffle rewrites apply to every scheme
fuse_bn_binarize = fuse_wbwtab_blocks  # first name of this pass
