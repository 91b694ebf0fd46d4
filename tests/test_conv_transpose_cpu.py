"""`QuantConvTranspose2d` on the CPU side (SURVEY 8 row f4): module surface / prepare() of all three schemes without a GPU, and
the evidence, recorded from the reference, that the reference's OWN wbwtab / dorefa classes are not runnable under current
PyTorch, which is why only the IAO one (IAO:510-636) has golden fixtures generated from the reference
(tests/golden/layer_iao_convT_*.npz) and the other two are pinned on the oracle's quantizers composed with ATen."""
import copy

import pytest
import torch
import torch.nn as nn

from tests.oracle_util import load_golden, rel_err


def _net():
    return nn.Sequential(nn.Conv2d(3, 16, 3, padding=1), nn.ReLU(), nn.ConvTranspose2d(16, 8, 4, stride=2, padding=1), nn.ReLU(),
                         nn.Conv2d(8, 4, 1))


def test_prepare_swaps_conv_transpose_in_every_scheme():
    from micronet_b200 import dorefa, iao, wbwtab
    base = _net()
    keys = list(base.state_dict().keys())
    d = dorefa.prepare(copy.deepcopy(base), a_bits=4, w_bits=4)
    assert isinstance(d[2], dorefa.QuantConvTranspose2d) and isinstance(d[2], nn.ConvTranspose2d)
    assert d[2].activation_quantizer.a_bits == 4 and d[2].weight_quantizer.w_bits == 4
    assert list(d.state_dict().keys()) == keys                      # stateless quantizers: no new keys (DF)
    w = wbwtab.prepare(copy.deepcopy(base), A=2, W=3)
    assert isinstance(w[2], wbwtab.QuantConvTranspose2d) and w[2].weight_quantizer.W == 3
    assert list(w.state_dict().keys()) == keys
    i = iao.prepare(copy.deepcopy(base))
    assert isinstance(i[2], iao.QuantConvTranspose2d)
    extra = set(i.state_dict().keys()) - set(keys)
    assert {"2.activation_quantizer.scale", "2.weight_quantizer.scale", "2.weight_quantizer.observer.min_val"} <= extra
    assert tuple(i[2].weight_quantizer.scale.shape) == (1,)         # per-layer observers whatever q_level says (IAO:552-560)
    for m in (d[2], w[2], i[2]):                                    # geometry carried over by name
        assert m.stride == (2, 2) and m.padding == (1, 1) and m.output_padding == (0, 0) and m.groups == 1 and m.dilation == (1, 1)
        assert m.weight.shape == base[2].weight.shape and m.weight.data_ptr() == m.weight.data_ptr()
    for m in (d[2], w[2], i[2]):                                    # no CPU path: the engine refuses CPU tensors loudly
        with pytest.raises(Exception):
            m(torch.randn(1, 16, 4, 4))


def test_reference_dorefa_and_wbwtab_conv_transpose_do_not_run():
    """what the reference's own classes did for QuantConvTranspose2d(8, 6, 3, stride=2, padding=1, output_padding=1),
    recorded by tests/golden/make_golden_convT_reference.py"""
    from micronet_b200 import dorefa, wbwtab
    from oracle import reference_port as O
    gold = load_golden("reference", "convT_modules")
    assert tuple(gold["dorefa.dilation"]) == (True, True)   # `bias` landed in `dilation` (DF:142-153 vs nn.ConvTranspose2d's argument order)
    for scheme in ("dorefa", "wbwtab"):
        err = str(gold[f"{scheme}.error"])
        assert err.startswith("TypeError") and "dilation" in err, err
    # the engine's modules take the same call with the geometry the reference meant
    for m in (dorefa.QuantConvTranspose2d(8, 6, 3, stride=2, padding=1, output_padding=1),
              wbwtab.QuantConvTranspose2d(8, 6, 3, stride=2, padding=1, output_padding=1)):
        assert m.dilation == (1, 1) and m.groups == 1 and m.bias is not None
        assert m.stride == (2, 2) and m.padding == (1, 1) and m.output_padding == (1, 1)
    # the IAO class is keyword-correct and runs: the oracle port reproduces its output
    iao = O.IaoQuantConvTranspose2d(8, 6, 3, stride=2, padding=1, output_padding=1)
    iao.load_state_dict({k[len("iao.init."):]: torch.from_numpy(v) for k, v in gold.items() if k.startswith("iao.init.")})
    y = iao(torch.from_numpy(gold["x"]))
    assert tuple(y.shape) == (2, 6, 10, 10)
    assert rel_err(y.detach(), gold["iao.y"]) <= 1e-6
