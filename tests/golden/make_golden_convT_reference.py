#!/usr/bin/env python
"""Record how the reference's own QuantConvTranspose2d classes behave under current PyTorch, for
tests/test_conv_transpose_cpu.py:

    python tests/golden/make_golden_convT_reference.py <path to a micronet checkout>

The DoReFa and wbwtab classes pass (dilation, groups, bias) positionally in the wrong order to
nn.ConvTranspose2d, so `bias` lands in `dilation` and their forward raises TypeError; the IAO class is
keyword-correct and runs.  The fixture keeps the DoReFa module's geometry, both errors, and the IAO
module's initial state, input and output (one training-mode forward)."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GEOM = dict(stride=2, padding=1, output_padding=1)   # QuantConvTranspose2d(8, 6, 3, **GEOM)


def main(ref):
    sys.path.insert(0, ref)
    import micronet.compression.quantization.wbwtab.quantize as ref_wb
    import micronet.compression.quantization.wqaq.dorefa.quantize as ref_df
    import micronet.compression.quantization.wqaq.iao.quantize as ref_iao

    torch.manual_seed(0)
    x = torch.randn(2, 8, 5, 5)
    out = {"x": x.numpy().copy()}
    df = ref_df.QuantConvTranspose2d(8, 6, 3, **GEOM)
    out["dorefa.dilation"] = np.array(df.dilation)
    out["dorefa.groups"] = np.array(df.groups)
    out["dorefa.has_bias"] = np.array(df.bias is not None)
    for name, mod in (("dorefa", df), ("wbwtab", ref_wb.QuantConvTranspose2d(8, 6, 3, **GEOM))):
        try:
            mod(x)
            out[f"{name}.error"] = np.array("")
        except Exception as e:
            out[f"{name}.error"] = np.array(f"{type(e).__name__}: {e}")
    iao = ref_iao.QuantConvTranspose2d(8, 6, 3, **GEOM)
    for n, t in iao.state_dict().items():
        out[f"iao.init.{n}"] = t.detach().clone().numpy()
    out["iao.y"] = iao(x).detach().numpy().copy()
    np.savez_compressed(os.path.join(HERE, "reference_convT_modules.npz"), **out)


if __name__ == "__main__":
    torch.set_num_threads(1)
    main(sys.argv[1])
