"""QAT step of NIN-GC prepared with ``wbwtab.prepare(A=2, W=3)`` WITHOUT ``fuse_bn`` (nn.BatchNorm2d + binarizer modules:
no producer writes a bf16 plane, so every wbwtab layer packs its own +-1 input) at batch 256 on cuda:0.

    python harness/unfused_wbwtab_step.py OUT [--steps 20 --warmup 5]     # img/s (eager steps), conv kernel totals -> OUT
    python harness/unfused_wbwtab_step.py --compare OUT_A OUT_B           # loss / gradients of two builds, rel <= 1e-5

OUT receives result.json (img/s of the timed steps, per-kind KernelTimer totals of one more step; a kind includes the
calls that found the shape outside the kernel's cover) and step.npz (loss and
gradients of one seeded forward + backward of the freshly initialised model).  --compare prints, per array, the relative
difference of the two builds."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from harness import train as H  # noqa: E402

BATCH, HW = 256, 32


def measure(out, steps, warmup):
    from micronet_b200 import _lib as L, functional as F_
    dev = torch.device("cuda:0")
    model = H.prepare_engine(H.build_float_model("nin_gc"), "wbwtab", W=3, A=2).to(dev).train()
    x, t = H.synthetic_batch(BATCH, HW, seed=100, device=dev)
    loss = torch.nn.functional.cross_entropy(model(x), t)
    loss.backward()
    arrays = {"loss": loss.detach().cpu().numpy()}
    arrays.update({f"grad.{n}": p.grad.detach().cpu().numpy() for n, p in model.named_parameters()})
    os.makedirs(out, exist_ok=True)
    np.savez(os.path.join(out, "step.npz"), **arrays)

    # eager steps: the un-fused graph does not capture into a CUDA graph (on either side of the comparison)
    stepper = H.QatStepper(model, lr=0.01, flat=True, graph=False)
    for i in range(warmup):
        stepper.step(x, t)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        stepper.step(x, t)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    F_.TIMER = F_.KernelTimer()
    stepper.step(x, t)
    torch.cuda.synchronize()
    kinds, layers = {}, {}
    for (kind, shape), times in F_.TIMER.summary().items():
        kinds[kind] = kinds.get(kind, 0.0) + sum(times)
        layers[f"{kind} {list(shape)}"] = sum(times)
    F_.TIMER = None
    L.tc_check()
    res = {"gpu": torch.cuda.get_device_name(dev), "batch": BATCH, "steps": steps, "ms_per_step": ms,
           "img_per_s": BATCH / (ms / 1e3), "conv_kernel_ms_per_step": dict(sorted(kinds.items())),
           "conv_kernel_ms_per_layer": layers}
    with open(os.path.join(out, "result.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


def _rel(x, y):
    x, y = x.astype(np.float64), y.astype(np.float64)
    return float(np.abs(x - y).max() / max(np.abs(y).max(), 1e-30))


def compare(da, db):
    a, b = np.load(os.path.join(da, "step.npz")), np.load(os.path.join(db, "step.npz"))
    worst = 0.0
    for k in a.files:
        rel = _rel(a[k], b[k])
        noise = k.endswith("conv.bias")     # in front of a training-mode BatchNorm: mathematically zero, rounding noise
        if not noise:
            worst = max(worst, rel)
        print(f"{k:32s} rel {rel:9.2e}{'  (noise: bias in front of a BatchNorm)' if noise else ''}")
    print(f"worst rel A vs B (without the conv biases) {worst:.2e}: {'OK' if worst <= 1e-5 else 'ABOVE 1e-5'}")
    return worst <= 1e-5


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("out", nargs="?")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--compare", nargs=2, metavar="DIR")
    args = ap.parse_args()
    if args.compare:
        sys.exit(0 if compare(*args.compare) else 1)
    measure(args.out, args.steps, args.warmup)
