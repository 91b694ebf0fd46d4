#!/usr/bin/env python
"""Headline benchmark: QAT-step images/sec on synthetic CIFAR-10-shaped batches.

    python bench.py --gpus 1 --steps 20 --warmup 5            # this repo's CUDA engine
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 2   # CPU reference path (oracle port)
    python bench.py --workload resnet18_iao_w8a8_bnfuse       # another BASELINE.json config as the measured workload
    python bench.py --steps 20 --dump-outputs DIR             # + what the last timed step computed, as DIR/<name>.npy

Workload (BASELINE.json configs[1]): NIN-GC, wbwtab W-ternary / A-binary, batch 256 per GPU,
3x32x32 inputs, CrossEntropy + Adam(lr 0.01) - the reference's training step
(wbwtab/main.py:70-98).  N > 1: one process per GPU under torchrun, batch sharded (256 per
rank, weak scaling), one NCCL all-reduce of the flat gradient bucket per step (PTQ inference,
configs[4]: independent replicas, no collective).

One JSON line on stdout (rank 0).  `value` is timed with inputs resident in HBM; `e2e` is the
same step fed from pinned HOST buffers (H2D of the batch + D2H of the loss / logits inside the timed
region); `roofline` is for the dominant engine kernel, timed live with CUDA events on the
launching stream; `cpu_baseline` is the oracle port of the reference timed on the host cores;
`extra_workloads` (N = 1 only) are short runs of the other BASELINE.json configs in the same process."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from harness import train as H  # noqa: E402

WORKLOAD = "nin_gc_wbwtab_w3a2"   # BASELINE.json configs[1]; --workload picks another config
BATCH_PER_GPU = 256
CPU_SAMPLE_BATCH = 32
DUMP_BYTES = 64 * 10**6   # --dump-outputs budget, .npy headers included
NAMES = {"nin_gc_wbwtab_w3a2": "NIN-GC wbwtab W-ternary/A-binary QAT step (BASELINE.json configs[1])",
         "nin_dorefa_w8a8": "NIN DoReFa W8A8 QAT step (configs[0] model)",
         "resnet18_iao_w8a8_bnfuse": "ResNet-18 IAO W8A8 per-channel + BN-fuse QAT step (configs[2])",
         "nin_gc_dorefa_w4a4": "NIN-GC DoReFa W4A4 QAT step (configs[3] model)",
         "resnet18_iao_ptq_224": "ResNet-18 IAO int8 PTQ inference forward (configs[4])"}


def metric_name(workload):
    return "ptq_inference_images_per_sec" if H.WORKLOADS[workload].get("inference") else "qat_step_images_per_sec"


def batch_per_gpu(workload):
    return H.WORKLOADS[workload].get("batch", BATCH_PER_GPU)


def cpu_sample_batch(workload):
    return 2 if H.WORKLOADS[workload].get("inference") else CPU_SAMPLE_BATCH


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops"], "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu, self.first = [], None, gpu_index, 0

    def mark(self):
        """samples before this point (warm-up) are not reported"""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        rows = self.rows[self.first:] or self.rows[-1:]
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def conv_algorithmic(shape, kind):
    """SURVEY.md §8(d): F = 2*B*K*P*Q*(C/g)*R*S ; Bytes = 4(B*C*H*W + B*K*P*Q) + 4|W| (fp32 module surface)."""
    B, C, Hh, W, K, R, S, sh, sw, ph, pw, dh, dw, G = shape
    P = (Hh + 2 * ph - dh * (R - 1) - 1) // sh + 1
    Q = (W + 2 * pw - dw * (S - 1) - 1) // sw + 1
    flops = 2.0 * B * K * P * Q * (C // G) * R * S
    nbytes = 4.0 * (B * C * Hh * W + B * K * P * Q) + 4.0 * K * (C // G) * R * S
    return flops, nbytes


def config_dict(workload, n_gpus, cpu_arm=False):
    w = H.WORKLOADS[workload]
    hw = w["hw"]
    if cpu_arm:
        # the CPU arm runs ONE host process on a bounded sample, whatever --gpus says: state exactly that
        b = cpu_sample_batch(workload)
        return {"workload": f"{NAMES[workload]}, synthetic 3x{hw}x{hw}, CPU sample batch {b} (same model, same step)",
                "global_batch": b, "per_gpu_batch": None, "parallelism": "1 host process",
                "note": "bounded CPU sample of the engine arm's workload; it does not scale with --gpus"}
    b = batch_per_gpu(workload)
    return {"workload": f"{NAMES[workload]}, synthetic 3x{hw}x{hw}, batch {b}/GPU",
            "global_batch": b * n_gpus, "per_gpu_batch": b,
            "optimizer": "none (inference)" if w.get("inference") else "Adam lr=0.01",
            "parallelism": f"{n_gpus} independent replicas" if w.get("inference") else f"dp{n_gpus}",
            "l2": "per-step activation working set >> 126 MB L2, 4 rotating input batches (no flush needed)"}


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own path (oracle port) on the host cores, bounded sample
# ----------------------------------------------------------------------------------------------------------
def run_cpu_baseline(workload, steps=3, warmup=2):
    ncpu = os.cpu_count() or 1
    w = H.WORKLOADS[workload]
    b = cpu_sample_batch(workload)
    model = H.prepare_oracle(H.build_float_model(w["model"]), w["scheme"], **w["prepare"])
    if w.get("inference"):
        stepper = H.InferStepper(model)
        stepper.calibrate([H.synthetic_batch(b, w["hw"], seed=50 + i)[0] for i in range(1)])
        what = "eval forward passes"
    else:
        stepper = H.QatStepper(model, lr=0.01, wd=w["wd"])
        what = "QAT steps"
    x, t = H.synthetic_batch(b, w["hw"], seed=1)
    # use as many host threads as actually help: at these batch sizes ATen's intra-op pool stops scaling
    # (and then collapses) well before 100+ threads, so probe a few pool sizes with one step each
    best, cores = None, 1
    for n in sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(n)
        stepper.step(x, t)
        t0 = time.perf_counter()
        stepper.step(x, t)
        d = time.perf_counter() - t0
        if best is None or d < best:
            best, cores = d, n
        if d > 2.5 * best:
            break
    torch.set_num_threads(cores)
    for _ in range(warmup):
        stepper.step(x, t)
    t0 = time.perf_counter()
    for _ in range(steps):
        stepper.step(x, t)
    dt = (time.perf_counter() - t0) / steps
    return {"value": b / dt, "unit": "img/s", "cores": cores, "kind": "port",
            "sample": f"{steps} {what} of the same model at batch {b} (oracle/reference_port.py, "
                      f"torch CPU, best of the probed thread counts = {cores} of {ncpu} host cores), {dt * 1e3:.0f} ms/step"}, dt


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    base, dt = run_cpu_baseline(wl, steps=max(1, args.steps), warmup=max(0, args.warmup))
    line = {"impl": "reference", "metric": metric_name(wl), "value": base["value"], "unit": "img/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": config_dict(wl, args.gpus, cpu_arm=True), "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# engine arm
# ----------------------------------------------------------------------------------------------------------
def dump_outputs(path, model, result, inference):
    """write what the last timed step handed its caller as <path>/<name>.npy (float32): the logits of an inference
    step; the loss of a QAT step with the parameters and floating-point buffers it updated and the gradients it
    computed.  Past DUMP_BYTES in all, every array is cut to the same fraction of its elements, a seeded random
    sample kept in index order (flattened), so that two builds fed the same arguments dump comparable arrays."""
    arrays = {"logits" if inference else "loss": result}
    if not inference:
        for n, p in model.named_parameters():
            arrays[f"param.{n}"] = p
            if p.grad is not None:
                arrays[f"grad.{n}"] = p.grad
        for n, b in model.named_buffers():
            if b.is_floating_point():
                arrays[f"buffer.{n}"] = b
    total = sum(a.numel() for a in arrays.values())
    keep = min(1.0, (DUMP_BYTES - 256 * len(arrays)) / 4 / total)   # 256 B: the header of one .npy file, and its one kept element
    os.makedirs(path, exist_ok=True)
    for i, (name, a) in enumerate(arrays.items()):
        a = a.detach().float().cpu()
        if keep < 1.0:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(i))[:max(1, int(a.numel() * keep))]
            a = a.flatten()[idx.sort().values]
        np.save(os.path.join(path, f"{name}.npy"), a.numpy())


def run_engine(workload, steps, warmup, dev, rank, world, detail, dump=None):
    """time `steps` steps of one workload; returns the measurement dict (rank-local, max over ranks for times).
    `dump`: directory that receives what the last timed step computed (rank 0)"""
    from micronet_b200 import _lib as L, functional as F_
    w = H.WORKLOADS[workload]
    inference = bool(w.get("inference"))
    B = batch_per_gpu(workload)
    model = H.prepare_engine(H.build_float_model(w["model"]), w["scheme"], **w["prepare"],
                             **w.get("engine_extra", {})).to(dev)
    nbuf = 4
    host = [H.synthetic_batch(B, w["hw"], seed=100 + rank * 17 + i, pin=True) for i in range(nbuf)]
    devb = [(x.to(dev), t.to(dev)) for x, t in host]
    if inference:
        stepper = H.InferStepper(model, graph=os.environ.get("MNB_GRAPH", "1") == "1")
        stepper.calibrate([devb[i][0][: max(2, B // 8)] for i in range(w.get("calib_batches", 2))])
    else:
        stepper = H.QatStepper(model, lr=0.01, wd=w["wd"], flat=True, graph=os.environ.get("MNB_GRAPH", "1") == "1")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, n):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            step_fn(i)
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    last = [None]

    def step_resident(i):
        x, t = devb[i % nbuf]
        last[0] = stepper.step(x, t).detach()   # a loss kept with its autograd graph would break the CUDA graph capture

    out_host = torch.empty((B, 10) if inference else (), dtype=torch.float32).pin_memory()

    def step_e2e(i):
        hx, ht = host[i % nbuf]
        x = hx.to(dev, non_blocking=True)
        t = ht.to(dev, non_blocking=True)
        res = stepper.step(x, t)
        out_host.copy_(res.detach(), non_blocking=False)  # D2H read of the step's result (loss / logits)

    sampler = ClockSampler(dev.index or 0) if detail and rank == 0 else None
    if sampler:
        sampler.start()  # started before the warm-up so that nvidia-smi is already streaming in the timed region
    for i in range(max(warmup, 5 if getattr(stepper, "graph_wanted", False) else 0)):
        step_resident(i)   # (a graph-replaying stepper captures after 3 eager steps: keep >= 2 replays in the warm-up)
    if sampler:
        sampler.mark()
    ms_total = timed(step_resident, steps)
    torch.cuda.synchronize()
    L.tc_check()   # a bounded pipeline wait that gave up would have produced garbage: fail loudly instead
    clocks = sampler.stop() if sampler else None
    if dump and rank == 0:
        dump_outputs(dump, model, last[0], inference)
    for i in range(2):
        step_e2e(i)
    ms_e2e = timed(step_e2e, steps)
    L.tc_check()
    # per-kernel CUDA-event timings and the launch count come from an adjacent EAGER pass of the same stepper (a replayed
    # graph runs the same kernels without going through the Python wrappers that place the events)
    graph_used = getattr(stepper, "graph", None) is not None
    saved = (getattr(stepper, "graph", None), getattr(stepper, "graph_wanted", False))
    if hasattr(stepper, "graph"):
        stepper.graph, stepper.graph_wanted = None, False
    timer = None
    for i in range(2):
        step_resident(i)   # eager allocations after a capture come from the non-graph pool: let the caching allocator fill it
    torch.cuda.synchronize()
    launches0 = L.launch_count()
    dsteps = min(steps, 3)
    if detail:
        F_.TIMER = F_.KernelTimer()
    ms_detail = timed(step_resident, dsteps)
    torch.cuda.synchronize()
    timer, F_.TIMER = F_.TIMER, None
    launches = (L.launch_count() - launches0) * steps // dsteps
    if hasattr(stepper, "graph"):
        stepper.graph, stepper.graph_wanted = saved
    imgs = B * world * steps
    res = {"workload": workload, "metric": metric_name(workload), "value": imgs / (ms_total / 1e3), "unit": "img/s",
           "ms_per_step": ms_total / steps, "steps": steps, "warmup": warmup, "per_gpu_batch": B,
           "e2e": {"value": imgs / (ms_e2e / 1e3), "unit": "img/s", "ms_per_step": ms_e2e / steps,
                   "h2d_bytes_per_step": (B * 3 * w["hw"] * w["hw"] * 4 + B * 8) * world,
                   "d2h_bytes_per_step": (B * 10 * 4 if inference else 4) * world},
           "gpu_launches": int(launches), "clocks": clocks, "timer": timer,
           "ms_total": ms_detail,   # the eager detail pass the per-kernel events were recorded in (dsteps steps)
           "detail_steps": dsteps,
           "cuda_graph": {"used": bool(graph_used), "error": getattr(stepper, "graph_error", None),
                          "eager_ms_per_step": ms_detail / dsteps}}
    del stepper, model
    torch.cuda.empty_cache()
    return res


def kernel_table(timer, ms_total, steps, hbm, tfl):
    agg = {}
    for (kind, shape), times in timer.summary().items():
        agg[(kind, shape)] = (sum(times), len(times))
    rows = []
    for (kind, shape), (tot, n) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
        fl, nb = conv_algorithmic(shape, kind)
        t_roof = max(nb / (hbm * 1e9), fl / (tfl * 1e12))
        rows.append({"kind": kind, "shape": list(shape), "launches": n, "avg_us": tot / n * 1e3,
                     "algo_GBps": nb / (tot / n / 1e3) / 1e9, "algo_TFLOPs": fl / (tot / n / 1e3) / 1e12,
                     "hbm_roof_us": nb / (hbm * 1e9) * 1e6, "roof_us": t_roof * 1e6,
                     "frac_of_roof": t_roof / (tot / n / 1e3)})
    return agg, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--kernels-json", default=None, help="dump the per-kernel CUDA-event timings of the timed region")
    ap.add_argument("--workload", default=WORKLOAD, choices=sorted(H.WORKLOADS),
                    help="default: the headline configuration (BASELINE.json configs[1])")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step of the workload computed to DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return main_reference(args)
    args.warmup = max(args.warmup, 3)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the engine has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    wl = args.workload
    main_res = run_engine(wl, args.steps, args.warmup, dev, rank, world, detail=True, dump=args.dump_outputs)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm, tfl, peak_src = _peaks()
    timer, ms_total, dsteps = main_res.pop("timer"), main_res.pop("ms_total"), main_res.pop("detail_steps")
    # kernel time per step (CUDA events of the eager detail pass) over the TIMED step (graph replay): the eager pass itself is
    # longer than the step it repeats (Python / ctypes issue time between launches), so it is not the denominator
    step_ms = main_res["ms_per_step"]
    agg, rows = kernel_table(timer, ms_total, args.steps, hbm, tfl)
    if args.kernels_json:
        json.dump({"ms_per_step": main_res["ms_per_step"], "kernels": rows}, open(args.kernels_json, "w"), indent=1)
    roof = None
    if agg:
        # dominant engine kernel by total device time
        (dk, dshape), (dtot, dn) = max(agg.items(), key=lambda kv: kv[1][0])
        flops, nbytes = conv_algorithmic(dshape, dk)
        avg_s = dtot / dn / 1e3
        t_hbm, t_tc = nbytes / (hbm * 1e9), flops / (tfl * 1e12)
        if t_hbm >= t_tc:
            roof = {"bound": "hbm", "achieved": nbytes / avg_s / 1e9, "peak": hbm, "unit": "GB/s"}
        else:
            roof = {"bound": "tensor", "achieved": flops / avg_s / 1e12, "peak": tfl, "unit": "TFLOP/s"}
        roof["frac"] = roof["achieved"] / roof["peak"]
        traffic = tsrc = None
        tpath = os.path.join(ROOT, "profiles", "kernel_traffic.json")
        if os.path.exists(tpath):  # measured dram__bytes_{read,write}.sum per launch from the committed ncu capture
            tj = json.load(open(tpath))
            rec = tj["kernels"].get(f"{dk}:{list(dshape)}")
            traffic = rec["dram_bytes"] if rec else None
            tsrc = tj.get("source")
        t_roof_sum = sum(max(conv_algorithmic(sh, k)[1] / (hbm * 1e9), conv_algorithmic(sh, k)[0] / (tfl * 1e12)) * n
                         for (k, sh), (_, n) in agg.items())
        roof.update({"traffic": traffic, "traffic_source": tsrc, "algorithmic_bytes": nbytes, "algorithmic_flops": flops,
                     "peak_source": peak_src,
                     "kernel": f"conv2d_{dk} shape(B,C,H,W,K,R,S,sh,sw,ph,pw,dh,dw,G)={list(dshape)}",
                     "avg_launch_us": avg_s * 1e6, "launches_timed": dn, "share_of_step": dtot / dsteps / step_ms,
                     "engine_conv_share_of_step": sum(v[0] for v in agg.values()) / dsteps / step_ms,
                     # all engine conv launches of the timed region: sum of their rooflines / sum of their measured times
                     "all_conv_kernels_frac": t_roof_sum * 1e3 / max(1e-9, sum(v[0] for v in agg.values()))})
    line = {"metric": main_res["metric"], "value": main_res["value"], "unit": "img/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f32 (bf16 tensor-core products of exact integer levels / exact bf16 pieces, fp32 accumulate)",
            "data": "synthetic", "config": config_dict(wl, world), "clocks": main_res["clocks"], "e2e": main_res["e2e"],
            "gpu_launches": main_res["gpu_launches"], "cuda_graph": main_res["cuda_graph"], "roofline": roof}
    if world == 1 and not args.no_extra:
        # the other BASELINE.json configs, a few steps each, so that the driver-run record covers them too
        extras = []
        for name in H.WORKLOADS:
            if name == wl:
                continue
            try:
                r = run_engine(name, 5, 3, dev, rank, world, detail=True)
                t2, ms2, ds2 = r.pop("timer"), r.pop("ms_total"), r.pop("detail_steps")
                agg2, _ = kernel_table(t2, ms2, 5, hbm, tfl)
                r.pop("clocks")
                r["config"] = config_dict(name, world)["workload"]
                r["engine_conv_share_of_step"] = sum(v[0] for v in agg2.values()) / ds2 / r["ms_per_step"] if agg2 else None
                r["conv_kinds"] = sorted({k for k, _ in agg2})
                extras.append(r)
            except Exception as e:  # an extra must never take the headline line down with it
                extras.append({"workload": name, "error": f"{type(e).__name__}: {e}"[:300]})
        line["extra_workloads"] = extras
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"], _ = run_cpu_baseline(wl)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
