"""Fused BatchNorm2d + binarizer (micronet_b200.fused) against nn.BatchNorm2d (fp64, CPU) followed by the
oracle's binarizer (WB:11-36 / WB:79-94): outputs, saturate-STE gradients, parameter gradients, running stats."""
import copy

import pytest
import torch
import torch.nn as nn

from oracle import reference_port as O
from tests.oracle_util import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"

SHAPES = [  # B, C, H, W  (NIN-GC planes + ragged ones that take the scalar kernels)
    (8, 192, 32, 32), (8, 96, 16, 16), (16, 192, 8, 8), (3, 10, 1, 1), (5, 7, 3, 5), (2, 33, 6, 6), (64, 160, 32, 32),
]


def _pair(c, seed):
    torch.manual_seed(seed)
    bn = nn.BatchNorm2d(c)
    with torch.no_grad():
        bn.weight.copy_(torch.rand(c) + 0.5)
        bn.bias.copy_(torch.randn(c) * 0.3)
        bn.running_mean.copy_(torch.randn(c) * 0.1)
        bn.running_var.copy_(torch.rand(c) + 0.5)
    return bn


def _reference(bn, x, go, groups=1, pool=False):
    """fp64 BatchNorm + the oracle's binarizer [+ 2x2 max-pool] [+ channel shuffle]; returns y, bn output, dx, dgamma, dbeta"""
    ref = copy.deepcopy(bn).double()
    xr = x.double().requires_grad_(True)
    pre = ref(xr)
    y = O.wb_binarize_activation(pre)
    if pool:
        y = nn.functional.max_pool2d(y, 2, 2)
    if groups > 1:
        y = _shuffle(y, groups)
    y.backward(go.double())
    return y.detach(), pre.detach(), xr.grad, ref.weight.grad, ref.bias.grad, ref


def _shuffle(x, groups):
    """nin_gc.py:9-21"""
    b, c, h, w = x.shape
    return x.view(b, groups, c // groups, h, w).transpose(1, 2).contiguous().view(b, c, h, w)


def _groups_for(c):
    return next(g for g in (4, 3, 2, 11, 5, 7, 1) if c % g == 0)


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("shuffled", [False, True], ids=["plain", "shuffled"])
def test_fused_bn_binarize_matches_bn_then_oracle_binarizer(shape, training, shuffled):
    from micronet_b200.fused import BatchNormBinarize2d
    B, C, H, W = shape
    groups = _groups_for(C) if shuffled else 1
    bn = _pair(C, sum(shape))
    bn.train(training)
    x = torch.randn(B, C, H, W) * 1.5 + 0.2
    go = torch.randn(B, C, H, W)
    # sign() and the saturate STE are discontinuous at bn = 0 and |bn| = 1: move the few elements that sit
    # within fp32 rounding of those points away from them, so the comparison below can be strict
    for _ in range(6):
        with torch.no_grad():
            pre = copy.deepcopy(bn).double()(x.double())
        edge = (pre.abs() < 1e-4) | ((pre.abs() - 1).abs() < 1e-4)
        if not edge.any():
            break
        x = torch.where(edge, x + 0.01, x)
    assert not edge.any()
    y_r, pre, dx_r, dg_r, db_r, ref = _reference(bn, x, go, groups)

    fused = BatchNormBinarize2d(C)
    fused.load_state_dict(bn.state_dict())
    fused = fused.to(DEV).train(training)
    fused.out_shuffle_groups = groups
    xg = x.to(DEV).requires_grad_(True)
    y = fused(xg)
    y.backward(go.to(DEV))
    # the by-product handed to the producing convolution: channel sums of dx

    assert torch.equal(y.detach().cpu().double(), y_r)
    assert rel_err(xg.grad, dx_r) < 1e-5
    assert rel_err(fused.weight.grad, dg_r) < 1e-5 and rel_err(fused.bias.grad, db_r) < 1e-5
    if training:
        assert rel_err(fused.running_mean, ref.running_mean) < 1e-6
        assert rel_err(fused.running_var, ref.running_var) < 1e-6
        assert int(fused.num_batches_tracked) == int(ref.num_batches_tracked) == 1
    else:
        assert torch.equal(fused.running_mean.cpu(), bn.running_mean)


POOLED = [(8, 256, 32, 32), (8, 64, 16, 16), (4, 32, 8, 8), (3, 12, 4, 24), (2, 33, 6, 6), (2, 6, 10, 12)]  # last two: two-step path


@pytest.mark.parametrize("shape", POOLED, ids=[str(s) for s in POOLED])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("shuffled", [False, True], ids=["plain", "shuffled"])
def test_fused_bn_binarize_pool_matches_reference_chain(shape, training, shuffled):
    """BatchNorm -> binarizer -> MaxPool2d(2, 2) [-> shuffle] in one module: +-1 windows are all ties, so the
    first-maximum rule decides which input receives the pooled gradient"""
    from micronet_b200.fused import BatchNormBinarize2d
    B, C, H, W = shape
    groups = _groups_for(C) if shuffled else 1
    bn = _pair(C, sum(shape) + 1)
    bn.train(training)
    x = torch.randn(B, C, H, W) * 1.5 + 0.2
    go = torch.randn(B, C, H // 2, W // 2)
    for _ in range(6):
        with torch.no_grad():
            pre = copy.deepcopy(bn).double()(x.double())
        edge = (pre.abs() < 1e-4) | ((pre.abs() - 1).abs() < 1e-4)
        if not edge.any():
            break
        x = torch.where(edge, x + 0.01, x)
    assert not edge.any()
    y_r, pre, dx_r, dg_r, db_r, ref = _reference(bn, x, go, groups, pool=True)
    fused = BatchNormBinarize2d(C)
    fused.load_state_dict(bn.state_dict())
    fused = fused.to(DEV).train(training)
    fused.out_shuffle_groups, fused.pool2 = groups, True
    xg = x.to(DEV).requires_grad_(True)
    y = fused(xg)
    y.backward(go.to(DEV))
    assert torch.equal(y.detach().cpu().double(), y_r)
    assert rel_err(xg.grad, dx_r) < 1e-5
    assert rel_err(fused.weight.grad, dg_r) < 1e-5 and rel_err(fused.bias.grad, db_r) < 1e-5
    if training:
        assert rel_err(fused.running_mean, ref.running_mean) < 1e-6 and rel_err(fused.running_var, ref.running_var) < 1e-6


def test_bn_sign_backward_hands_over_channel_sums_of_dx():
    """conv(bias) -> fused BN: the bias gradient comes from the BN backward's by-product; it must equal the
    channel sums of the dx the kernel wrote (pure rounding noise for a training-mode BN: compare to |dx| scale)"""
    from micronet_b200.fused import BNSignFn
    torch.manual_seed(5)
    B, C, H, W = 16, 48, 16, 16
    x = (torch.randn(B, C, H, W) * 2).to(DEV).requires_grad_(True)
    gamma, beta = (torch.rand(C) + 0.5).to(DEV).requires_grad_(True), torch.randn(C).to(DEV).requires_grad_(True)
    for training in (True, False):
        mean, var = x.detach().mean((0, 2, 3)), x.detach().var((0, 2, 3), unbiased=False)
        y = BNSignFn.apply(x, gamma, beta, mean, torch.rsqrt(var + 1e-5), training, 1, False)
        captured = {}

        def grab(g, captured=captured):
            captured["sum"] = getattr(g, "_mnb_channel_sum", None)

        handle = x.register_hook(grab)
        x.grad = None
        y.backward(torch.randn_like(y))
        handle.remove()
        assert captured["sum"] is not None
        want = x.grad.double().sum((0, 2, 3))
        scale = x.grad.double().abs().sum((0, 2, 3))
        assert ((captured["sum"].double() - want).abs() <= 1e-6 * scale + 1e-12).all()


POOLS = [  # B, C, H, W, k, s, p, shuffle groups
    (4, 64, 32, 32, 2, 2, 0, 1), (4, 64, 16, 16, 2, 2, 0, 4), (3, 30, 32, 32, 3, 2, 1, 1), (3, 30, 17, 19, 3, 2, 1, 3),
    (2, 8, 9, 9, 3, 1, 1, 1), (2, 6, 10, 14, 2, 2, 0, 2), (2, 5, 7, 7, 2, 2, 0, 1), (2, 4, 12, 12, 3, 3, 0, 2),
]


@pytest.mark.parametrize("cfg", POOLS, ids=[str(c) for c in POOLS])
@pytest.mark.parametrize("binary", [True, False], ids=["pm1", "float"])
def test_engine_maxpool_is_bit_identical_to_aten(cfg, binary):
    """+-1 inputs are all ties: the first-maximum rule decides where the gradient goes"""
    from micronet_b200.fused import EngineMaxPool2d
    B, C, H, W, k, s, p, g = cfg
    torch.manual_seed(sum(cfg))
    x = torch.randn(B, C, H, W)
    if binary:
        x = torch.where(x < 0, -torch.ones_like(x), torch.ones_like(x))
    xe = x.to(DEV).requires_grad_(True)
    xr = x.to(DEV).requires_grad_(True)
    pool = EngineMaxPool2d(k, s, p)
    pool.out_shuffle_groups = g
    y = pool(xe)
    yr = nn.functional.max_pool2d(xr, k, s, p)
    if g > 1:
        yr = _shuffle(yr, g)
    assert torch.equal(y, yr)
    go = torch.randn_like(yr)
    y.backward(go)
    yr.backward(go)
    assert torch.equal(xe.grad, xr.grad)


def test_fused_model_step_matches_unfused_engine_model():
    """whole NIN-GC step, fused vs unfused engine models: same loss and (up to sign flips at |bn| ~ 0)
    the same gradients"""
    import micronet_b200 as E
    from harness import models as zoo
    torch.manual_seed(1)
    base = zoo.NINGC()
    zoo.init_like_reference(base)
    x = torch.randn(16, 3, 32, 32).to(DEV)
    t = torch.randint(0, 10, (16,)).to(DEV)
    out = {}
    for name, kw in (("plain", {}), ("fused", {"fuse_bn": True})):
        m = E.wbwtab.prepare(base, A=2, W=3, **kw).to(DEV).train()
        loss = nn.functional.cross_entropy(m(x), t)
        loss.backward()
        out[name] = (loss.item(), {n: p.grad.clone() for n, p in m.named_parameters()},
                     {n: b.clone() for n, b in m.named_buffers()})
    assert abs(out["plain"][0] - out["fused"][0]) < 2e-3 * abs(out["plain"][0])
    # a binarized net amplifies the handful of sign flips at |bn| ~ 1e-7 layer by layer, so deep tensors are
    # compared by direction; the first fused block sees bit-identical inputs and is compared tightly
    first = "model.0.bn"
    for key in ("running_mean", "running_var"):
        assert rel_err(out["fused"][2][f"{first}.{key}"], out["plain"][2][f"{first}.{key}"]) < 1e-5, first
    flat = {k: torch.cat([g.flatten() for g in out[k][1].values()]).double() for k in out}
    cos = torch.dot(flat["plain"], flat["fused"]) / (flat["plain"].norm() * flat["fused"].norm())
    assert cos > 0.98, float(cos)


def test_dorefa_fuse_option_agrees_with_the_unfused_engine():
    """pool kernels are bit-identical to ATen and a folded shuffle is only an addressing change; since round 2 the fuse
    option also merges BatchNorm2d + ReLU + the next conv's activation quantizer into one producer
    (fused.BatchNormReluQuant2d), whose BatchNorm arithmetic (one fma, statistics from mnb_bn_batch_stats) differs from
    ATen's in the last bit: a few activation levels land on the other side of a rounding tie, so the fused model agrees
    with the unfused engine model in direction and loss, not bit for bit (the strict per-module checks are
    tests/test_gpu_fused_dorefa.py)."""
    import micronet_b200 as E
    from harness import models as zoo
    torch.manual_seed(2)
    base = zoo.NINGC()
    zoo.init_like_reference(base)
    x = torch.randn(8, 3, 32, 32).to(DEV)
    t = torch.randint(0, 10, (8,)).to(DEV)
    out = {}
    for name, kw in (("plain", {}), ("fused", {"fuse": True})):
        m = E.dorefa.prepare(base, a_bits=4, w_bits=4, **kw).to(DEV).train()
        loss = nn.functional.cross_entropy(m(x), t)
        loss.backward()
        out[name] = (loss.detach().clone(), {n: p.grad.clone() for n, p in m.named_parameters()})
    assert abs(out["plain"][0].item() - out["fused"][0].item()) <= 2e-3 * max(1.0, abs(out["plain"][0].item()))
    for n, g in out["plain"][1].items():
        if n.endswith("conv.bias"):
            continue      # a conv bias in front of a training-mode BatchNorm has a mathematically zero gradient: noise
        a, b = out["fused"][1][n].flatten().double(), g.flatten().double()
        assert torch.dot(a, b) / (a.norm() * b.norm()) > 0.99, n


@pytest.mark.parametrize("cfg", [(8, 256, 256, 32, 1, 2, 2), (8, 256, 512, 16, 3, 16, 1), (4, 512, 512, 16, 1, 4, 4)],
                         ids=["1x1g2", "3x3g16", "1x1g4"])
@pytest.mark.parametrize("pool", [False, True], ids=["plain", "pooled"])
def test_wbwtab_layer_between_two_fused_producers_on_the_packed_operand_family(cfg, pool):
    """BatchNormBinarize2d -> wbwtab QuantConv2d -> BatchNormBinarize2d with both conv operands written by the producers
    (+-1 plane forward: mnb_bn_sign_fwd_packed, gradient pieces backward: mnb_bn_sign_bwd_pack) against the same chain on the
    generic kernels (MNB_PK=off), which the oracle tests pin: identical +-1 outputs, gradients to 1e-5 (weight gradient:
    plus the cancellation allowance of tests/test_gpu_parity.py).  ``pool``: the consuming producer has the 2x2 max-pool folded
    in (mnb_bn_sign_pool_bwd_pack writes the full-resolution gradient pieces)."""
    import micronet_b200 as E
    from micronet_b200 import _lib as L
    from micronet_b200.fused import BatchNormBinarize2d
    from tests.test_gpu_parity import _cancellation_allowance
    B, C, K, H, R, G, sg = cfg
    torch.manual_seed(sum(cfg))
    x = torch.randn(B, C, H, H) * 1.3
    go = torch.randn(B, K, H // 2, H // 2) if pool else torch.randn(B, K, H, H)
    bn0, bn1 = _pair(C, 3), _pair(K, 4)
    conv = E.wbwtab.QuantConv2d(C, K, R, padding=R // 2, groups=G, W=3)
    res = {}
    for mode in ("off", "auto"):
        L.PK_MODE = mode
        try:
            p0 = BatchNormBinarize2d(C); p0.load_state_dict(bn0.state_dict()); p0.out_shuffle_groups = sg
            p1 = BatchNormBinarize2d(K); p1.load_state_dict(bn1.state_dict()); p1.pool2 = pool
            cv = copy.deepcopy(conv)
            net = nn.Sequential(p0, cv, p1).to(DEV).train()
            captured = {}
            cv.register_forward_hook(lambda m, i, o: captured.__setitem__("y", o.detach().clone()))
            xg = x.to(DEV).requires_grad_(True)
            out = net(xg)
            out.backward(go.to(DEV))
            torch.cuda.synchronize()
            res[mode] = dict(out=out.detach().cpu(), conv=captured["y"].cpu(), dx=xg.grad.cpu(), dw=cv.weight.grad.cpu(),
                             db=cv.bias.grad.cpu(), dg1=p1.weight.grad.cpu(), db1=p1.bias.grad.cpu(), dg0=p0.weight.grad.cpu())
        finally:
            L.PK_MODE = "auto"
    a, b = res["off"], res["auto"]
    assert rel_err(b["conv"], a["conv"]) <= 1e-6                      # integer-level products: exact up to the bias add
    flips = (a["out"] != b["out"]).float().mean().item()
    assert flips <= 1e-4, flips                                         # sign of bn values within rounding of 0
    for k in ("dx", "dg1", "db1", "dg0"):
        assert rel_err(b[k], a[k]) <= 2e-5 if flips else rel_err(b[k], a[k]) <= 1e-5, (k, rel_err(b[k], a[k]))
    allow = _cancellation_allowance(go, 1.0) / a["dw"].abs().max().item()
    assert rel_err(b["dw"], a["dw"]) <= 1e-5 + 50 * allow, (rel_err(b["dw"], a["dw"]), allow)
    assert b["db"].abs().max().item() <= 1e-4 * a["dw"].abs().max().item() + a["db"].abs().max().item() * 2 + 1e-6
    L.tc_check()


@pytest.mark.parametrize("shape", [(8, 1024, 8, 8, 10, 1), (4, 256, 16, 16, 24, 3)], ids=["head1x1", "3x3"])
def test_unquantized_conv_behind_a_binarizer_runs_on_the_packed_family(shape):
    """fused.EnginePmConv2d (the fp32 10-way head of a wbwtab model, WB:247-331 leaves it un-quantized): BatchNorm+binarizer
    -> conv on the packed-operand family (+-1 plane from the producer, exact pieces of the fp32 weights) against ATen in
    fp64 on the same +-1 tensor; without the +-1 tag the module is exactly the stock convolution."""
    import torch.nn.functional as TF
    from micronet_b200 import _lib as L, functional as F_
    from micronet_b200.fused import BatchNormBinarize2d, EnginePmConv2d
    B, C, H, W, K, R = shape
    torch.manual_seed(sum(shape))
    bn = BatchNormBinarize2d(C).to(DEV).train()
    conv = EnginePmConv2d(C, K, R, padding=R // 2).to(DEV)
    x = (torch.randn(B, C, H, W) * 1.5).to(DEV)
    go = torch.randn(B, K, H, W).to(DEV)
    F_.TIMER = F_.KernelTimer()
    try:
        a = bn(x)
        a.retain_grad()
        y = conv(a)
        y.backward(go)
        torch.cuda.synchronize()
        kinds = {k for k, _, _, _ in F_.TIMER.records}
    finally:
        F_.TIMER = None
    L.tc_check()
    assert {"fwd_pk", "dgrad_pk", "wgrad_pk"} <= kinds, kinds
    ad = a.detach().double().cpu().requires_grad_(True)
    wd = conv.weight.detach().double().cpu().requires_grad_(True)
    bd = conv.bias.detach().double().cpu().requires_grad_(True)
    yd = TF.conv2d(ad, wd, bd, 1, R // 2)
    yd.backward(go.double().cpu())
    assert rel_err(y.detach(), yd.detach()) <= 2e-6
    assert rel_err(a.grad, ad.grad) <= 1e-5
    assert rel_err(conv.weight.grad, wd.grad) <= 1e-5
    assert rel_err(conv.bias.grad, bd.grad) <= 1e-5
    plain = torch.randn(B, C, H, W, device=DEV)          # no +-1 tag: the stock path, bit for bit
    assert torch.equal(conv(plain), TF.conv2d(plain, conv.weight, conv.bias, 1, R // 2))


@pytest.mark.parametrize("shape", [(4, 256, 32, 32, 256, 1, 2, 2), (4, 512, 8, 8, 1024, 3, 32, 4)], ids=["1x1", "3x3"])
def test_plane_only_producer_gives_the_same_block(shape):
    """BatchNormBinarize2d.plane_only (fuse pass: the only reader is a conv of the packed-operand family): the fp32 output is
    never written, functional.materialized() rebuilds it from the bf16 plane, and conv output / every gradient are
    bit-identical to the run that writes it."""
    from micronet_b200 import _lib as L, functional as F_
    from micronet_b200.fused import BatchNormBinarize2d
    B, C, H, W, K, R, G, sg = shape
    torch.manual_seed(sum(shape))
    x0 = (torch.randn(B, C, H, W) * 1.5).to(DEV)
    w_int = torch.randint(-1, 2, (K, C // G, R, R), dtype=torch.int16).to(DEV)
    w_scale = (torch.rand(K) * 0.02 + 0.001).to(DEV)
    go = torch.randn(B, K, H, W).to(DEV)
    res = {}
    for flag in (False, True):
        torch.manual_seed(5)
        bn = BatchNormBinarize2d(C).to(DEV).train()
        bn.out_shuffle_groups, bn.plane_only = sg, flag
        x = x0.clone().requires_grad_(True)
        wq = (w_int.float() * w_scale.view(-1, 1, 1, 1)).requires_grad_(True)
        a = bn(x)
        assert bool(getattr(a, "_mnb_plane_only", False)) == flag
        vals = F_.materialized(a).detach().clone()
        out = F_.quant_conv2d(a, wq, None, w_int, w_scale, None, (1, 1), (R // 2, R // 2), (1, 1), G)
        out.backward(go)
        res[flag] = (vals, out.detach(), x.grad, wq.grad, bn.weight.grad, bn.bias.grad)
    L.tc_check()
    for a, b in zip(res[True], res[False]):
        assert torch.equal(a, b)


# B, C, H, W, K, R, groups, shuffle groups of the producer
PLANE_CASES = [(4, 256, 32, 32, 256, 1, 2, 1), (4, 256, 32, 32, 256, 1, 2, 2), (4, 512, 16, 16, 512, 1, 4, 16),
               (5, 1024, 8, 8, 1024, 1, 8, 32), (4, 256, 16, 16, 512, 3, 16, 2), (4, 512, 8, 8, 1024, 3, 32, 4),
               (3, 64, 16, 16, 32, 3, 1, 1)]


@pytest.mark.parametrize("case", PLANE_CASES, ids=[str(c) for c in PLANE_CASES])
def test_packed_producer_and_conv_match_the_unpacked_path(case):
    """The producer's bf16 operand plane (y._mnb_pk_pm1, mnb_bn_sign_fwd_packed) is exactly the +-1 output in
    [B][C/8][H][W][8] order (the producer's OUTPUT channel order), and the convolution fed by it equals an fp64 convolution
    of the fp32 tensor."""
    import torch.nn.functional as TF
    from micronet_b200 import _lib as L, functional as F_
    from micronet_b200.fused import BatchNormBinarize2d
    B, C, H, W, K, R, G, sg = case
    torch.manual_seed(sum(case))
    bn = BatchNormBinarize2d(C).to(DEV).train()
    bn.out_shuffle_groups = sg
    with torch.no_grad():
        bn.weight.copy_(torch.rand(C) + 0.5)
        bn.bias.copy_(torch.randn(C) * 0.3)
    x = (torch.randn(B, C, H, W) * 1.5).to(DEV)
    y = bn(x)
    plane = getattr(y, "_mnb_pk_pm1", None)
    assert plane is not None, "producer did not emit the packed operand"
    want = y.detach().view(B, C // 8, 8, H, W).permute(0, 1, 3, 4, 2).contiguous().to(torch.bfloat16).flatten()
    assert torch.equal(plane.view(torch.bfloat16), want)
    w_int = torch.randint(-1, 2, (K, C // G, R, R), dtype=torch.int16).to(DEV)
    w_scale = (torch.rand(K) * 0.02 + 0.001).to(DEV)
    bias = torch.randn(K).to(DEV)
    wq = w_int.float() * w_scale.view(-1, 1, 1, 1)
    out = F_.quant_conv2d(y, wq, bias, w_int, w_scale, None, (1, 1), (R // 2, R // 2), (1, 1), G)
    L.tc_check()
    ref = TF.conv2d(y.detach().double().cpu(), wq.double().cpu(), bias.double().cpu(), 1, R // 2, 1, G)
    assert rel_err(out.detach(), ref) < 2e-6


@pytest.mark.parametrize("case", PLANE_CASES[:5], ids=[str(c) for c in PLANE_CASES[:5]])
def test_block_with_packed_forward_has_the_same_gradients(case):
    """BatchNorm+binarizer -> conv on the packed-operand family with producer-written operands (the default) against the
    generic kernels (MNB_PK=off).  Same +-1 operand in the forward: identical outputs; gradients agree to the accuracy of the
    backward's operand split."""
    from micronet_b200 import _lib as L, functional as F_
    from micronet_b200.fused import BatchNormBinarize2d
    B, C, H, W, K, R, G, sg = case
    torch.manual_seed(sum(case) + 1)
    x0 = (torch.randn(B, C, H, W) * 1.5).to(DEV)
    w_int = torch.randint(-1, 2, (K, C // G, R, R), dtype=torch.int16).to(DEV)
    w_scale = (torch.rand(K) * 0.02 + 0.001).to(DEV)
    go = torch.randn(B, K, H, W).to(DEV)
    res = {}
    for mode in ("off", "auto"):
        L.PK_MODE = mode
        try:
            torch.manual_seed(5)
            bn = BatchNormBinarize2d(C).to(DEV).train()
            bn.out_shuffle_groups = sg
            x = x0.clone().requires_grad_(True)
            wq = (w_int.float() * w_scale.view(-1, 1, 1, 1)).requires_grad_(True)
            F_.TIMER = F_.KernelTimer()
            out = F_.quant_conv2d(bn(x), wq, None, w_int, w_scale, None, (1, 1), (R // 2, R // 2), (1, 1), G)
            out.backward(go)
            torch.cuda.synchronize()
            kinds = {k for k, _, _, _ in F_.TIMER.records}
            res[mode] = (out.detach(), x.grad, wq.grad, bn.weight.grad, kinds)
        finally:
            L.PK_MODE = "auto"
            F_.TIMER = None
    assert not any(k.endswith("_pk") for k in res["off"][4]), res["off"][4]
    assert {"fwd_pk", "dgrad_pk", "wgrad_pk"} <= res["auto"][4], res["auto"][4]
    assert rel_err(res["auto"][0], res["off"][0]) <= 1e-6
    for a, b in zip(res["auto"][1:4], res["off"][1:4]):
        assert rel_err(a, b) <= 1e-5     # two-piece dy operand (MNB_PK_TERMS_BWD=2): ~3e-6, inside the 1e-5 contract
    L.tc_check()
