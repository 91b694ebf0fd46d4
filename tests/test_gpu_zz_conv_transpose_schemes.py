"""dorefa / wbwtab `QuantConvTranspose2d` (DF:125-174, WB:198-244; SURVEY 8 row f4).  The reference's own classes cannot serve as
the oracle here: they pass (dilation, groups, bias) positionally in the wrong order to nn.ConvTranspose2d and their forward raises
TypeError under current PyTorch (tests/test_conv_transpose_cpu.py keeps that evidence, recorded from the reference).  The engine
modules implement the intent, so the check is the composition of the ORACLE's quantizers (pinned by the golden fixtures) with
ATen's conv_transpose2d on the CPU."""
import pytest
import torch
import torch.nn.functional as TF

from tests.oracle_util import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Cin, Cout, k, stride, pad, output_padding, B, H
GEOMS = [(64, 32, 4, 2, 1, 0, 4, 16), (32, 64, 3, 2, 1, 1, 3, 8)]


@pytest.mark.parametrize("geom", GEOMS, ids=[str(g) for g in GEOMS])
@pytest.mark.parametrize("bits", [(8, 8), (4, 4)], ids=["w8a8", "w4a4"])
def test_dorefa_conv_transpose_matches_the_oracle_composition(geom, bits):
    from micronet_b200 import dorefa
    from oracle import reference_port as O
    ci, co, k, st, pad, op, B, H = geom
    ab, wb = bits
    torch.manual_seed(ci + co + ab)
    m = dorefa.QuantConvTranspose2d(ci, co, k, stride=st, padding=pad, output_padding=op, a_bits=ab, w_bits=wb)
    with torch.no_grad():
        m.weight.mul_(3.0)
        m.bias.uniform_(-0.5, 0.5)
    w0, b0 = m.weight.detach().clone(), m.bias.detach().clone()
    x = torch.relu(torch.randn(B, ci, H, H)) * 4
    m.to(DEV).train()
    xe = x.to(DEV).requires_grad_(True)
    ye = m(xe)
    go = torch.randn(ye.shape)
    ye.backward(go.to(DEV))
    xo, wo, bo = x.clone().requires_grad_(True), w0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    yo = TF.conv_transpose2d(O.dorefa_quantize_activation(xo, ab), O.dorefa_quantize_weight(wo, wb), bo, st, pad, op, 1, 1)
    yo.backward(go)
    assert rel_err(ye.detach(), yo.detach()) <= 1e-5
    assert rel_err(xe.grad, xo.grad) <= 1e-5
    assert rel_err(m.weight.grad, wo.grad) <= 1e-5
    assert rel_err(m.bias.grad, bo.grad) <= 1e-5


@pytest.mark.parametrize("geom", GEOMS, ids=[str(g) for g in GEOMS])
@pytest.mark.parametrize("W", [2, 3], ids=["binary", "ternary"])
def test_wbwtab_conv_transpose_matches_the_oracle_composition(geom, W):
    from micronet_b200 import wbwtab
    from oracle import reference_port as O
    ci, co, k, st, pad, op, B, H = geom
    torch.manual_seed(ci + co + W)
    m = wbwtab.QuantConvTranspose2d(ci, co, k, stride=st, padding=pad, output_padding=op, W=W)
    with torch.no_grad():
        m.weight.mul_(6.0)
        m.bias.uniform_(-0.5, 0.5)
    w0, b0 = m.weight.detach().clone(), m.bias.detach().clone()
    x = torch.where(torch.randn(B, ci, H, H) < 0, -1.0, 1.0)
    m.to(DEV).train()
    xe = x.to(DEV).requires_grad_(True)
    ye = m(xe)
    go = torch.randn(ye.shape)
    ye.backward(go.to(DEV))
    xo, bo = x.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    wo = torch.nn.Parameter(w0.clone())          # W = 2 mean-centres and clamps the parameter in place (WB:98-102)
    yo = TF.conv_transpose2d(xo, O.wb_quantize_weight(wo, W), bo, st, pad, op, 1, 1)
    yo.backward(go)
    assert rel_err(ye.detach(), yo.detach()) <= 1e-5
    assert rel_err(xe.grad, xo.grad) <= 1e-5
    assert rel_err(m.weight.grad, wo.grad) <= 1e-5
    assert rel_err(m.bias.grad, bo.grad) <= 1e-5
    assert rel_err(m.weight.detach(), wo.detach()) <= 1e-6      # the in-place mutation, if any, is the same
