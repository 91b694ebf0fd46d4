"""Packed-operand tensor-core family (csrc/mnb_pk.cu) against fp64 convolutions of the same operands.

Integer operands must reproduce the fp64 result exactly (every product and partial sum is an integer below 2^24);
fp32 operands split into three bf16 pieces must agree to fp32 rounding (<= 2e-6 of the largest result)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as TF

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# B, C, H, W, K, R, stride, pad, groups
SHAPES = [
    (3, 64, 32, 32, 64, 3, 1, 1, 1),      # ResNet conv2_x
    (3, 64, 32, 32, 128, 3, 2, 1, 1),     # ResNet conv3_1 (stride 2)
    (3, 64, 32, 32, 128, 1, 2, 0, 1),     # ResNet 1x1 stride-2 shortcut
    (5, 128, 16, 16, 128, 3, 1, 1, 1),    # ResNet conv3_x
    (4, 256, 8, 8, 512, 3, 2, 1, 1),      # ResNet conv5_1
    (7, 512, 4, 4, 512, 3, 1, 1, 1),      # ResNet conv5_x: 4x4 images, several per tile, 4 N tiles
    (2, 3, 32, 32, 64, 3, 1, 1, 1),       # 3-channel stem
    (2, 96, 16, 16, 192, 5, 1, 2, 1),     # NIN 5x5
    (2, 192, 8, 8, 192, 3, 1, 1, 1),      # NIN 3x3
    (2, 192, 32, 32, 160, 1, 1, 0, 1),    # NIN 1x1, N = 160
    (2, 160, 32, 32, 96, 1, 1, 0, 1),
    (2, 192, 8, 8, 10, 1, 1, 0, 1),       # 10-way head
    (2, 256, 16, 16, 512, 3, 1, 1, 16),   # NIN-GC grouped 3x3
    (2, 256, 32, 32, 256, 1, 1, 0, 2),    # NIN-GC grouped 1x1
    (1, 16, 24, 224, 32, 3, 1, 1, 1),     # wide image: column tiles
    (1, 3, 64, 64, 16, 7, 2, 3, 1),       # 7x7 stride-2 stem
    (2, 32, 9, 9, 48, 3, 1, 0, 1),        # 'valid' padding, odd size
    (9, 512, 1, 1, 10, 1, 1, 0, 1),       # linear layer view
    (4, 512, 16, 16, 512, 1, 1, 0, 4),    # NIN-GC grouped 1x1, 4 groups
    (4, 512, 8, 8, 1024, 3, 1, 1, 32),    # NIN-GC grouped 3x3, 32 groups
    (5, 1024, 8, 8, 1024, 1, 1, 0, 8),    # NIN-GC grouped 1x1, 8 groups, odd batch
    (3, 48, 4, 4, 64, 1, 1, 0, 1),        # 4x4 images, 1x1
    (2, 16, 12, 12, 16, 3, 1, 1, 1),      # W not a power of two
    (2, 32, 16, 16, 32, 5, 1, 2, 1),      # 5x5, 32 channels
]
IDS = ["x".join(map(str, s)) for s in SHAPES]


def _sh(shape):
    from micronet_b200 import _lib as L
    B, Cc, H, W, K, R, st, pad, G = shape
    return L.ConvShape(B, Cc, H, W, K, R, R, st, st, pad, pad, 1, 1, G)


def _ints(shape, gen, lim_x=127, lim_w=127):
    B, Cc, H, W, K, R, st, pad, G = shape
    x = torch.randint(-lim_x, lim_x + 1, (B, Cc, H, W), generator=gen).float()
    w = torch.randint(-lim_w, lim_w + 1, (K, Cc // G, R, R), generator=gen).float()
    return x, w


def _ref(x, w, shape, bias=None):
    B, Cc, H, W, K, R, st, pad, G = shape
    return TF.conv2d(x.double(), w.double(), None if bias is None else bias.double(), st, pad, 1, G)


def _unpack(planes, terms, B, Cc, H, W):
    c8 = (Cc + 7) // 8
    t = planes.view(torch.bfloat16).view(terms, B, c8, H, W, 8).float().sum(0)
    return t.permute(0, 1, 4, 2, 3).reshape(B, c8 * 8, H, W)[:, :Cc]


def test_pack_act_planes_hold_exact_pieces():
    from micronet_b200 import pk as PK
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(3, 19, 6, 10, generator=g) * 3).to(DEV)
    for terms in (1, 2, 3):
        planes, _ = PK.pack_act(x, None, terms)
        back = _unpack(planes, terms, 3, 19, 6, 10)
        err = (back - x).abs().max().item() / x.abs().max().item()
        assert err <= (2.0 ** -8, 2.0 ** -16, 0.0)[terms - 1] * 1.01, (terms, err)
    sc = (torch.rand(19, generator=g) + 0.5).to(DEV)
    planes, _ = PK.pack_act(x, None, 3, ch_scale=sc)
    assert torch.equal(_unpack(planes, 3, 3, 19, 6, 10), x * sc.view(1, -1, 1, 1))
    # phase split: octet (h%2*2 + w%2)*C8 + c/8 of an [H/2, W/2] plane
    planes, _ = PK.pack_act(x, None, 3, phase_split=True)
    ph = planes.view(torch.bfloat16).view(3, 3, 4, 3, 3, 5, 8).float().sum(0)      # [b][phase][c8][h/2][w/2][8]
    for a in range(2):
        for b in range(2):
            got = ph[:, a * 2 + b].permute(0, 1, 4, 2, 3).reshape(3, 24, 3, 5)[:, :19]
            assert torch.equal(got, x[:, :, a::2, b::2])


@pytest.mark.parametrize("mode", ["dorefa4", "dorefa8", "iao_sym", "iao_asym"])
def test_pack_act_quantizer_matches_the_standalone_kernel(mode):
    from micronet_b200 import _lib as L, functional as F_, pk as PK
    g = torch.Generator().manual_seed(11)
    x = (torch.randn(2, 24, 8, 8, generator=g) * 4).to(DEV)
    if mode.startswith("dorefa"):
        spec = F_.ActSpec(L.ACT_DOREFA, bits=int(mode[6:]))
        terms, scale, zp = 1, 1.0 / (2 ** int(mode[6:]) - 1), 0.0
    else:
        sym = mode == "iao_sym"
        s = torch.tensor([0.037], device=DEV)
        z = torch.tensor([0.0 if sym else -101.0], device=DEV)
        lo, hi = torch.tensor([-4.5], device=DEV), torch.tensor([4.9], device=DEV)
        spec = F_.ActSpec(L.ACT_IAO, bits=8, qmin=-128 if sym else 0, qmax=127 if sym else 255, q_type=0 if sym else 1,
                          scale=s, zero_point=z, obs_min=lo, obs_max=hi)
        terms, scale, zp = (1 if sym else 2), 0.037, z.item()
    codes, bits, xq = F_.act_quant_raw(x, spec, True, True, True)
    qp = spec.struct()
    planes, bits8 = PK.pack_act(x, qp, terms, want_bits=True)
    lev = _unpack(planes, terms, 2, 24, 8, 8)
    want = codes.float() + spec.code_offset + zp
    assert torch.equal(lev, want)
    # STE flags: bit j of bits8[b, c/8, h, w] = flat NCHW bit of channel 8*(c/8) + j
    flat = bits.view(torch.int32)
    idx = torch.arange(x.numel(), device=DEV)
    passed = ((flat[idx // 32] >> (idx % 32)) & 1).view(x.shape).bool()
    got = torch.stack([(bits8 >> j) & 1 for j in range(8)], dim=2).reshape(2, 24, 8, 8).bool()
    assert torch.equal(got, passed)


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_forward_integer_operands_are_exact(shape):
    from micronet_b200 import _lib as L, pk as PK
    B, Cc, H, W, K, R, st, pad, G = shape
    g = torch.Generator().manual_seed(abs(hash(shape)) % (1 << 31))
    lim = 127 if Cc // G * R * R <= 1024 else 31          # keep |sum| < 2^24
    x, w = _ints(shape, g, lim, lim)
    x, w = x.to(DEV), w.to(DEV)
    sh = _sh(shape)
    assert PK.supported(sh, 0, 1, 1)
    x_pk, _ = PK.pack_act(x, None, 1, phase_split=st == 2)
    img = PK.pack_weight(sh, 0, 1, 1, w_int=w.to(torch.int16))
    ref = _ref(x, w, shape)
    y = torch.full(ref.shape, float("nan"), dtype=torch.float32, device=DEV)
    L.check(PK.conv(sh, 0, x_pk, 1, img, 1, y), "pk_conv")
    torch.cuda.synchronize()
    L.tc_check()
    assert torch.equal(y.double(), ref), (y.double() - ref).abs().max().item()


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_forward_fp32_operands_scale_and_bias(shape):
    from micronet_b200 import _lib as L, pk as PK
    B, Cc, H, W, K, R, st, pad, G = shape
    g = torch.Generator().manual_seed(abs(hash(shape)) % (1 << 31) + 1)
    x = (torch.randn(B, Cc, H, W, generator=g) * 2).to(DEV)
    w = (torch.randn(K, Cc // G, R, R, generator=g) * 0.1).to(DEV)
    bias = torch.randn(K, generator=g).to(DEV)
    nsc = (torch.rand(K, generator=g) + 0.5).to(DEV)
    sh = _sh(shape)
    x_pk, _ = PK.pack_act(x, None, 3, phase_split=st == 2)
    img = PK.pack_weight(sh, 0, 3, 3, w_f32=w)
    ref = _ref(x, w, shape) * (0.25 * nsc.double()).view(1, -1, 1, 1) + bias.double().view(1, -1, 1, 1)
    y = torch.full(ref.shape, float("nan"), dtype=torch.float32, device=DEV)
    L.check(PK.conv(sh, 0, x_pk, 3, img, 3, y, n_scale=nsc, a_scale_const=0.25, bias=bias), "pk_conv")
    torch.cuda.synchronize()
    L.tc_check()
    err = (y.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err <= 3e-6, err


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_data_gradient_with_ste_mask(shape):
    from micronet_b200 import _lib as L, pk as PK
    B, Cc, H, W, K, R, st, pad, G = shape
    g = torch.Generator().manual_seed(abs(hash(shape)) % (1 << 31) + 2)
    P, Q = (H + 2 * pad - R) // st + 1, (W + 2 * pad - R) // st + 1
    dy = torch.randn(B, K, P, Q, generator=g).to(DEV)
    w_int = torch.randint(-127, 128, (K, Cc // G, R, R), generator=g, dtype=torch.int16).to(DEV)
    w_scale = (torch.rand(K, generator=g) * 0.02 + 0.001).to(DEV)
    w_scale[0] = 0.0                       # a dead channel must contribute nothing
    wq = w_int.double() * w_scale.double().view(-1, 1, 1, 1)
    ref = torch.nn.grad.conv2d_input((B, Cc, H, W), wq, dy.double(), st, pad, 1, G)
    sh = _sh(shape)
    assert PK.supported(sh, 1, 3, 1)
    dy_pk, _ = PK.pack_act(dy, None, 3, ch_scale=w_scale)
    img = PK.pack_weight(sh, 1, 3, 1, w_int=w_int, kzero=w_scale)
    use_mask = G == 1 or (Cc // G) % 8 == 0
    bits8 = None
    if use_mask:
        bits8 = torch.randint(0, 256, (B, (Cc + 7) // 8, H, W), generator=g, dtype=torch.uint8).to(DEV)
        keep = torch.stack([(bits8 >> j) & 1 for j in range(8)], dim=2).reshape(B, -1, H, W)[:, :Cc].double()
        ref = ref * keep * 0.1
    dx = torch.full((B, Cc, H, W), float("nan"), dtype=torch.float32, device=DEV)
    L.check(PK.conv(sh, 1, dy_pk, 3, img, 1, dx, bits8=bits8, gain=0.1 if use_mask else 1.0), "pk_conv dgrad")
    torch.cuda.synchronize()
    L.tc_check()
    err = (dx.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err <= 3e-6, err


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
@pytest.mark.parametrize("kind", ["levels", "fp32"])
def test_weight_gradient(shape, kind):
    from micronet_b200 import _lib as L, pk as PK
    B, Cc, H, W, K, R, st, pad, G = shape
    g = torch.Generator().manual_seed(abs(hash(shape)) % (1 << 31) + 3)
    P, Q = (H + 2 * pad - R) // st + 1, (W + 2 * pad - R) // st + 1
    dy = torch.randn(B, K, P, Q, generator=g).to(DEV)
    sh = _sh(shape)
    if not PK.wgrad_supported(sh, 3, 1):
        pytest.skip("outside the cover of the packed weight-gradient kernel")
    if kind == "levels":
        x = torch.randint(-128, 128, (B, Cc, H, W), generator=g).float().to(DEV)
        tx = 1
        a_scale = torch.tensor([0.031], device=DEV)
        kdiv = (torch.rand(K, generator=g) + 0.5).to(DEV)
        dy_pk, _ = PK.pack_act(dy, None, 3, ch_scale=kdiv)
        mul = 0.031
    else:
        x = (torch.randn(B, Cc, H, W, generator=g) * 2).to(DEV)
        tx, a_scale, kdiv, mul = 3, None, None, 1.0
        dy_pk, _ = PK.pack_act(dy, None, 3)
    x_pk, _ = PK.pack_act(x, None, tx, phase_split=st == 2)
    ref = torch.nn.grad.conv2d_weight(x.double(), (K, Cc // G, R, R), dy.double(), st, pad, 1, G) * mul
    dw = torch.full((K, Cc // G, R, R), float("nan"), dtype=torch.float32, device=DEV)
    L.check(PK.wgrad(sh, dy_pk, 3, x_pk, tx, dw, a_scale=a_scale, kdiv=kdiv), "pk_wgrad")
    torch.cuda.synchronize()
    L.tc_check()
    err = (dw.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err <= 3e-6, err


@pytest.mark.parametrize("shape", [(64, 64, 32, 32, 64, 3, 1, 1, 1), (128, 256, 8, 8, 256, 3, 1, 1, 1)], ids=["conv2_x", "conv4_x"])
def test_weight_gradient_long_reduction(shape):
    """65536 / 8192 positions: the reduction is cut into short tensor-core chains (the accumulator truncates)"""
    from micronet_b200 import _lib as L, pk as PK
    B, Cc, H, W, K, R, st, pad, G = shape
    g = torch.Generator().manual_seed(77)
    dy = torch.randn(B, K, H, W, generator=g).to(DEV)
    x = torch.randint(0, 256, (B, Cc, H, W), generator=g).float().to(DEV)
    sh = _sh(shape)
    dy_pk, _ = PK.pack_act(dy, None, 3)
    x_pk, _ = PK.pack_act(x, None, 1)
    ref = torch.nn.grad.conv2d_weight(x.double(), (K, Cc, R, R), dy.double(), st, pad, 1, G)
    dw = torch.empty((K, Cc, R, R), dtype=torch.float32, device=DEV)
    L.check(PK.wgrad(sh, dy_pk, 3, x_pk, 1, dw), "pk_wgrad")
    torch.cuda.synchronize()
    L.tc_check()
    err = (dw.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err <= 5e-6, err


def test_module_path_uses_the_packed_family_for_resnet_shapes():
    """QuantConv2dFn end to end (IAO symmetric quantizer, stride 2) against the generic CUDA-core kernels"""
    from micronet_b200 import _lib as L, functional as F_
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(4, 64, 16, 16, generator=g) * 2).to(DEV)
    w_int = torch.randint(-127, 128, (128, 64, 3, 3), generator=g, dtype=torch.int16).to(DEV)
    w_scale = (torch.rand(128, generator=g) * 0.02 + 0.001).to(DEV)
    wq = w_int.float() * w_scale.view(-1, 1, 1, 1)
    bias = torch.randn(128, generator=g).to(DEV)
    s, z = torch.tensor([0.04], device=DEV), torch.tensor([0.0], device=DEV)
    lo, hi = torch.tensor([-5.0], device=DEV), torch.tensor([5.1], device=DEV)
    spec = F_.ActSpec(L.ACT_IAO, bits=8, qmin=-128, qmax=127, q_type=0, scale=s, zero_point=z, obs_min=lo, obs_max=hi)
    gy = torch.randn(4, 128, 8, 8, generator=g).to(DEV)
    res = {}
    for mode in ("auto", "off"):
        L.PK_MODE = mode
        try:
            F_.TIMER = F_.KernelTimer()
            xg, wg = x.clone().requires_grad_(True), wq.clone().requires_grad_(True)
            y = F_.quant_conv2d(xg, wg, bias, w_int, w_scale, spec, (2, 2), (1, 1), (1, 1), 1)
            y.backward(gy)
            torch.cuda.synchronize()
            kinds = {k for k, _, _, _ in F_.TIMER.records}
            res[mode] = (y.detach(), xg.grad, wg.grad, kinds)
        finally:
            L.PK_MODE = "auto"
            F_.TIMER = None
    assert {"fwd_pk", "dgrad_pk", "wgrad_pk"} <= res["auto"][3], res["auto"][3]
    assert not any(k.endswith("_pk") for k in res["off"][3])
    for a, b, tol in zip(res["auto"][:3], res["off"][:3], (1e-6, 1e-5, 1e-5)):
        assert (a - b).abs().max().item() <= tol * b.abs().max().item()
    L.tc_check()
