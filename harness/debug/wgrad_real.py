"""debug: weight gradient of one wbwtab layer on the REAL tensors of a golden model step (oracle capture), through the
default dispatch, the packed-operand kernel with 3 and 2 gradient pieces and the CUDA-core kernel, each against an fp64
replay."""
import copy, sys
import torch
from tests.golden.cases import MODEL_CASES
from tests.oracle_util import load_golden, rel_err
from tests.test_gpu_parity import _zoo_model, _prepare_engine, DEV
from tests.test_oracle_golden import prepare_oracle
from micronet_b200 import _lib as L

name = "nin_gc_wb_binary"
case = next(c for c in MODEL_CASES if c["name"] == name)
gold = load_golden("model", name)
init = {k[5:]: torch.from_numpy(v) for k, v in gold.items() if k.startswith("init.")}
om = _zoo_model(case); om.load_state_dict(init); om = prepare_oracle(om, case); om.train()
em = _zoo_model(case); em.load_state_dict(init); em = _prepare_engine(em, case).to(DEV); em.train()
pristine = copy.deepcopy(om)
x, t = torch.from_numpy(gold["s0.x"]), torch.from_numpy(gold["s0.t"])
cap = {}
for n in ("model.4.conv", "model.8.conv"):
    mod = dict(om.named_modules())[n]
    def h(mod, inp, out, n=n):
        rec = {"x": inp[0].detach().clone()}
        cap[n] = rec
        out.register_hook(lambda g: rec.__setitem__("go", g.detach().clone()))
    mod.register_forward_hook(h)
torch.nn.functional.cross_entropy(om(x), t).backward()
for n, c in cap.items():
    go, xi = c["go"], c["x"]
    a = go.abs()
    print(f"{n}: go max {a.max():.2e} median {a.median():.2e} zeros {(a == 0).float().mean():.2f} per-image max {[f'{v:.1e}' for v in a.amax((1,2,3)).tolist()]}"
          f" per-channel max range {a.amax((0,2,3)).min():.1e}..{a.amax((0,2,3)).max():.1e}  x values {sorted(set(xi.flatten().tolist()))[:4]}")
    o64 = copy.deepcopy(dict(pristine.named_modules())[n]).double()
    xo = xi.double().clone().requires_grad_(True)
    o64(xo).backward(go.double())
    ref = o64.weight.grad
    for tag, setup in (("default", dict()), ("generic", dict(PK_MODE="off")), ("pk3", dict(PK_MODE="all", PK_TERMS_BWD=3)), ("pk2", dict(PK_MODE="all", PK_TERMS_BWD=2))):
        saved = {k: getattr(L, k) for k in setup}
        for k, v in setup.items(): setattr(L, k, v)
        try:
            e = copy.deepcopy(dict(em.named_modules())[n])
            xe = xi.to(DEV).requires_grad_(True)
            e(xe).backward(go.to(DEV))
            print(f"   {tag:9s} dW vs f64 {rel_err(e.weight.grad, ref):.2e}   dx vs f64 {rel_err(xe.grad, xo.grad):.2e}")
        finally:
            for k, v in saved.items(): setattr(L, k, v)
    # the same with the gradient rescaled to O(1): is it the magnitude?
    s = 1.0 / go.abs().max()
    e = copy.deepcopy(dict(em.named_modules())[n]); xe = xi.to(DEV).requires_grad_(True)
    e(xe).backward((go * s).to(DEV))
    print(f"   default with go scaled to max 1: dW vs f64 {rel_err(e.weight.grad / s, ref):.2e}")
L.tc_check()
