"""QuantConv2dFn's default dispatch (the tensor-core kernels) against the generic CUDA-core kernels (MNB_PK=off) and
ATen-CPU conv2d: forward, data gradient and weight gradient of the NIN-GC / NIN / ResNet layer shapes."""
import numpy as np
import pytest
import torch
import torch.nn.functional as TF

from tests.oracle_util import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# B, C, H, W, K, R, groups           (stride 1, 'same' padding)
SHAPES = [
    (4, 256, 32, 32, 256, 1, 2),     # NIN-GC conv 2/3
    (4, 256, 16, 16, 512, 3, 16),    # NIN-GC conv 4
    (4, 512, 16, 16, 512, 1, 4),     # NIN-GC conv 5/6
    (4, 512, 8, 8, 1024, 3, 32),     # NIN-GC conv 7
    (5, 1024, 8, 8, 1024, 1, 8),     # NIN-GC conv 8 (odd batch: partial 2-image tile)
    (3, 192, 32, 32, 160, 1, 1),     # NIN conv 2
    (2, 64, 32, 32, 64, 3, 1),       # ResNet conv2_x
    (2, 32, 16, 16, 32, 5, 1),       # 5x5
    (3, 48, 4, 4, 64, 1, 1),         # 4x4 images, 8 per tile
    (2, 16, 12, 12, 16, 3, 1),       # W not a power of two
]


def _run(x, wq, bias, w_int, w_scale, spec, R, G, pk_mode, pm1):
    from micronet_b200 import _lib as L, functional as F_
    L.PK_MODE = pk_mode
    try:
        xg = x.clone().requires_grad_(True)
        xg._mnb_pm1 = pm1     # +-1 input (a binarizer's output without a producer-written plane)
        y = F_.quant_conv2d(xg, wq, bias, w_int, w_scale, spec, (1, 1), (R // 2, R // 2), (1, 1), G)
        torch.cuda.synchronize()
        return y
    finally:
        L.PK_MODE = "auto"


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
@pytest.mark.parametrize("mode", ["raw_pm1", "raw_fp32", "dorefa8", "dorefa4", "iao_sym", "iao_asym"])
def test_tc_forward_matches_generic_and_cpu(shape, mode):
    from micronet_b200 import _lib as L, functional as F_
    B, C, H, W, K, R, G = shape
    g = torch.Generator().manual_seed(hash((shape, mode)) % (1 << 31))
    if mode == "raw_pm1":
        x = torch.randint(0, 2, (B, C, H, W), generator=g).float() * 2 - 1
    else:
        x = torch.randn(B, C, H, W, generator=g) * 3
    lim = 1 if mode.startswith("raw") else (255 if mode == "dorefa8" else (15 if mode == "dorefa4" else 127))
    w_int = torch.randint(-lim, lim + 1, (K, C // G, R, R), generator=g, dtype=torch.int16)
    w_scale = torch.rand(K, generator=g) * 0.02 + 0.001
    wq = w_int.float() * w_scale.view(-1, 1, 1, 1)
    bias = torch.randn(K, generator=g)
    spec = None
    bufs = {}
    if mode.startswith("dorefa"):
        spec = F_.ActSpec(L.ACT_DOREFA, bits=int(mode[6:]))
    elif mode.startswith("iao"):
        sym = mode == "iao_sym"
        qmin, qmax = (-128, 127) if sym else (0, 255)
        mn, mx = torch.tensor([-7.5]), torch.tensor([8.25])
        if sym:
            s = torch.max(mn.abs(), mx.abs()) / 127.5
            zp = torch.zeros(1)
        else:
            s = (mx - mn) / 255.0
            zp = torch.sign(mn) * torch.floor((mn / s).abs() + 0.5)
        bufs = {k: v.to(DEV) for k, v in dict(scale=s, zero_point=zp, obs_min=mn, obs_max=mx).items()}
        spec = F_.ActSpec(L.ACT_IAO, qmin=qmin, qmax=qmax, q_type=0 if sym else 1, **bufs)
    xd, wqd, bd, wid, wsd = (t.to(DEV) for t in (x, wq, bias, w_int, w_scale))
    err = L.tc_err_flag(torch.device(DEV))
    err.zero_()
    n0 = L.launch_count()
    y_tc = _run(xd, wqd, bd, wid, wsd, spec, R, G, "auto", mode == "raw_pm1")
    assert err.item() == 0, f"tensor-core pipeline timed out, code {err.item()}"
    y_gen = _run(xd, wqd, bd, wid, wsd, spec, R, G, "off", mode == "raw_pm1")
    assert torch.isfinite(y_tc).all()
    # both paths are exact on integer levels; on raw fp32 they differ only by fp32 summation order
    assert rel_err(y_tc, y_gen) <= (5e-6 if mode == "raw_fp32" else 1e-6), f"tc vs generic {rel_err(y_tc, y_gen)}"
    # CPU reference: conv2d of the dequantized operands
    if spec is None:
        xq = x
    else:
        _, _, xqd = F_.act_quant_raw(xd, spec, False, False, True)
        xq = xqd.cpu()
    want = TF.conv2d(xq.double(), wq.double(), bias.double(), 1, R // 2, 1, G).float()
    assert rel_err(y_tc, want) <= 1e-5, f"tc vs cpu {rel_err(y_tc, want)}"


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
@pytest.mark.parametrize("mode", ["raw", "dorefa8", "iao_sym"])
def test_tc_dgrad_matches_generic_and_cpu(shape, mode):
    """dx through the tensor-core data gradient (weight scale folded into dy, MNB_PK_TERMS_BWD pieces, fused STE)."""
    from micronet_b200 import _lib as L, functional as F_
    B, C, H, W, K, R, G = shape
    g = torch.Generator().manual_seed(hash((shape, mode, "dgrad")) % (1 << 31))
    x = torch.randn(B, C, H, W, generator=g) * 4
    lim = 1 if mode == "raw" else 127
    w_int = torch.randint(-lim, lim + 1, (K, C // G, R, R), generator=g, dtype=torch.int16)
    w_scale = torch.rand(K, generator=g) * 0.02 + 0.001
    wq = w_int.float() * w_scale.view(-1, 1, 1, 1)
    spec = None
    if mode == "dorefa8":
        spec = F_.ActSpec(L.ACT_DOREFA, bits=8)
    elif mode == "iao_sym":
        bufs = dict(scale=torch.tensor([9.0 / 127.5]), zero_point=torch.zeros(1), obs_min=torch.tensor([-9.0]),
                    obs_max=torch.tensor([7.0]))
        spec = F_.ActSpec(L.ACT_IAO, qmin=-128, qmax=127, q_type=0, **{k: v.to(DEV) for k, v in bufs.items()})
    go = torch.randn(B, K, H, W, generator=g)
    err = L.tc_err_flag(torch.device(DEV)); err.zero_()
    grads = {}
    for pk_mode in ("auto", "off"):
        L.PK_MODE = pk_mode
        try:
            xg = x.to(DEV).requires_grad_(True)
            y = F_.quant_conv2d(xg, wq.to(DEV), None, w_int.to(DEV), w_scale.to(DEV), spec, (1, 1), (R // 2, R // 2), (1, 1), G)
            y.backward(go.to(DEV))
            torch.cuda.synchronize()
            grads[pk_mode] = xg.grad.clone()
        finally:
            L.PK_MODE = "auto"
    assert err.item() == 0, f"tensor-core pipeline timed out, code {err.item()}"
    assert rel_err(grads["auto"], grads["off"]) <= 5e-6, rel_err(grads["auto"], grads["off"])
    # CPU: autograd of conv2d on the dequantized input
    from oracle import reference_port as O
    xr = x.clone().requires_grad_(True)
    if mode == "raw":
        xq = xr
    elif mode == "dorefa8":
        xq = O.dorefa_quantize_activation(xr, 8)
    else:
        s = torch.tensor([9.0 / 127.5])
        v = xr / s
        r = O._RoundRangeSTE.apply(v, torch.tensor([-9.0]) / s, torch.tensor([7.0]) / s, 0)
        xq = torch.clamp(r, -128, 127) * s
    TF.conv2d(xq, wq, None, 1, R // 2, 1, G).backward(go)
    assert rel_err(grads["auto"], xr.grad) <= 1e-5, rel_err(grads["auto"], xr.grad)


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
@pytest.mark.parametrize("mode", ["raw_pm1", "raw_fp32", "dorefa8", "iao_sym"])
def test_tc_wgrad_matches_generic_and_cpu(shape, mode):
    """dWq through the tensor-core weight gradient (MN-major operands, deterministic reduction over the batch);
    +-1 inputs are one exact bf16 piece, raw fp32 inputs MNB_PK_TERMS_BWD pieces."""
    from micronet_b200 import _lib as L, functional as F_
    from oracle import reference_port as O
    B, C, H, W, K, R, G = shape
    g = torch.Generator().manual_seed(hash((shape, mode, "wgrad")) % (1 << 31))
    if mode == "raw_pm1":
        x = torch.randint(0, 2, (B, C, H, W), generator=g).float() * 2 - 1
    else:
        x = torch.randn(B, C, H, W, generator=g) * 4
    lim = 1 if mode.startswith("raw") else 127
    w_int = torch.randint(-lim, lim + 1, (K, C // G, R, R), generator=g, dtype=torch.int16)
    w_scale = torch.rand(K, generator=g) * 0.02 + 0.001
    wq = w_int.float() * w_scale.view(-1, 1, 1, 1)
    spec = None
    if mode == "dorefa8":
        spec = F_.ActSpec(L.ACT_DOREFA, bits=8)
    elif mode == "iao_sym":
        bufs = dict(scale=torch.tensor([9.0 / 127.5]), zero_point=torch.zeros(1), obs_min=torch.tensor([-9.0]),
                    obs_max=torch.tensor([7.0]))
        spec = F_.ActSpec(L.ACT_IAO, qmin=-128, qmax=127, q_type=0, **{k: v.to(DEV) for k, v in bufs.items()})
    go = torch.randn(B, K, H, W, generator=g)
    err = L.tc_err_flag(torch.device(DEV)); err.zero_()
    grads = {}
    for pk_mode in ("auto", "off"):
        L.PK_MODE = pk_mode
        try:
            wg = wq.to(DEV).requires_grad_(True)
            xd = x.to(DEV)
            xd._mnb_pm1 = mode == "raw_pm1"
            y = F_.quant_conv2d(xd, wg, None, w_int.to(DEV), w_scale.to(DEV), spec, (1, 1), (R // 2, R // 2), (1, 1), G)
            y.backward(go.to(DEV))
            torch.cuda.synchronize()
            grads[pk_mode] = wg.grad.clone()
        finally:
            L.PK_MODE = "auto"
    assert err.item() == 0, f"tensor-core pipeline timed out, code {err.item()}"
    assert torch.isfinite(grads["auto"]).all()
    assert rel_err(grads["auto"], grads["off"]) <= 1e-5, rel_err(grads["auto"], grads["off"])
    if mode.startswith("raw"):
        xq = x
    elif mode == "dorefa8":
        xq = O.dorefa_quantize_activation(x, 8)
    else:
        s = torch.tensor([9.0 / 127.5])
        xq = torch.clamp(O.round_half_away(x / s), -128, 127) * s
    wr = wq.clone().double().requires_grad_(True)
    TF.conv2d(xq.double(), wr, None, 1, R // 2, 1, G).backward(go.double())
    assert rel_err(grads["auto"], wr.grad) <= 1e-5, rel_err(grads["auto"], wr.grad)
