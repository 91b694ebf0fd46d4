"""debug: accuracy of the tensor-core weight-gradient kernels against fp64 as a function of the gradient's conditioning
(random vs BatchNorm-backward-like: zero mean per channel, heavy tailed) for the two headline layer kinds."""
import os, sys
import torch
import torch.nn.functional as TF
from micronet_b200 import _lib as L, functional as F_
from tests.oracle_util import rel_err

DEV = "cuda:0"
torch.manual_seed(0)


def run(name, B, C, H, K, R, G, kind):
    x = (torch.randint(0, 2, (B, C, H, H)).float() * 2 - 1)
    w_int = torch.randint(-1, 2, (K, C // G, R, R), dtype=torch.int16)
    w_scale = torch.rand(K) * 0.02 + 0.001
    wq = w_int.float() * w_scale.view(-1, 1, 1, 1)
    go = torch.randn(B, K, H, H)
    if kind == "bn":      # like the gradient behind a BatchNorm: heavy tailed, zero mean and orthogonal to the conv output per channel
        go = go ** 3 * torch.rand(B, 1, 1, 1) * 4
        y = TF.conv2d(x, wq, None, 1, R // 2, 1, G)
        yh = (y - y.mean((0, 2, 3), keepdim=True)) / y.std((0, 2, 3), keepdim=True)
        go = go - go.mean((0, 2, 3), keepdim=True) - yh * (go * yh).mean((0, 2, 3), keepdim=True)
    wr = wq.clone().double().requires_grad_(True)
    TF.conv2d(x.double(), wr, None, 1, R // 2, 1, G).backward(go.double())
    w32 = wq.clone().requires_grad_(True)
    TF.conv2d(x, w32, None, 1, R // 2, 1, G).backward(go)
    cond = (TF.conv2d(x.abs().double().transpose(0, 1), go.abs().double().transpose(0, 1)[:K // G], None, 1, R // 2).max() / wr.grad.abs().max()).item() if G == 1 else float("nan")
    out = {}
    for tag, env in (("auto", {}), ("pk3", {"pk": 3}), ("pk2", {"pk": 2})):
        wg = wq.to(DEV).requires_grad_(True)
        if "pk" in env:
            L.PK_MODE, L.PK_TERMS_BWD = "all", env["pk"]
        else:
            L.PK_MODE = "auto"
        y = F_.quant_conv2d(x.to(DEV), wg, None, w_int.to(DEV), w_scale.to(DEV), None, (1, 1), (R // 2, R // 2), (1, 1), G)
        y.backward(go.to(DEV))
        out[tag] = rel_err(wg.grad, wr.grad)
    L.PK_MODE, L.PK_TERMS_BWD = "auto", 2
    print(f"{name:28s} B={B:3d} {kind:5s} cpu32 {rel_err(w32.grad, wr.grad):.1e}  " + "  ".join(f"{k} {v:.1e}" for k, v in out.items()) + f"  S/max {cond:.0f}")


for B in (8, 32):
    for kind in ("randn", "bn"):
        run("1x1 g2 256->256 @32", B, 256, 32, 256, 1, 2, kind)
        run("3x3 g16 256->512 @16", B, 256, 16, 512, 3, 16, kind)
        run("3x3 g32 512->1024 @8", B, 512, 8, 1024, 3, 32, kind)
        run("3x3 g1 64->64 @16", B, 64, 16, 64, 3, 1, kind)
L.tc_check()
