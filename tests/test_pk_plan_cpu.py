"""Host-side checks of the tensor-core kernels that need no GPU:

* every kernel that opts in to a large dynamic shared-memory budget stays inside the 227 KB per-block limit TOGETHER with its
  static shared memory (read from the built library with cuobjdump).  This is the check that would have caught the one failed
  GPU run of round 2 (gpurun call r3g: 2 KB of extra static shared memory in `pk_conv_kernel`, `cudaFuncSetAttribute: invalid
  argument` on every launch);
* the host-only plan of the packed-operand family (`mnb_pk_conv_plan`, `mnb_pk_wgrad_scratch_bytes`, `mnb_pk_wimage_bytes`,
  `mnb_pk_act_bytes`) covers every convolution of the BASELINE.json models at their bench shapes, inside shared / tensor memory,
  and every stride-1 layer with the operand pieces of a +-1 or raw fp32 input (functional.QuantConv2dFn's wbwtab layers)."""
import ctypes as C
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIMIT = 227 * 1024          # opt-in shared memory per block on sm_100
RESERVED = 1024             # per-block reservation that cuobjdump's SHARED figure includes

# kernel (mangled-name fragment) -> (source file, name of its dynamic shared-memory budget constant)
BUDGETS = {
    "pk14pk_conv_kernel": ("mnb_pk.cu", "kSmemBudget"),
    "pk15pk_wgrad_kernel": ("mnb_pk.cu", "kSmemBudget"),
    "tcfp3210fwd_kernel": ("mnb_conv_fp32_tc.cu", "kMaxDynSmem"),
    "tcfp3212wgrad_kernel": ("mnb_conv_fp32_tc.cu", "kMaxDynSmem"),
}


def _budget(src, name):
    text = open(os.path.join(ROOT, "micronet_b200", "csrc", src)).read()
    m = re.search(r"constexpr int %s = ([0-9*+\- ]+);" % name, text)
    assert m, (src, name)
    return int(eval(m.group(1)))      # e.g. "227 * 1024 - 3072"


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
def test_static_plus_dynamic_shared_memory_fits_the_block_limit():
    from micronet_b200 import _lib as L
    out = subprocess.run(["cuobjdump", "-res-usage", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = re.findall(r"Function (\S+?):\s*\n\s*(.*)", out)
    assert funcs, "cuobjdump printed no resource usage"
    seen = set()
    for name, usage in funcs:
        m = re.search(r"SHARED:(\d+)", usage)
        static = max(0, int(m.group(1)) - RESERVED) if m else 0
        for frag, (src, const) in BUDGETS.items():
            if frag in name:
                seen.add(frag)
                dyn = _budget(src, const)
                assert static + dyn <= LIMIT, f"{name}: static {static} + dynamic budget {dyn} > {LIMIT}"
        regs = re.search(r"REG:(\d+)", usage)
        assert regs and int(regs.group(1)) <= 255
    assert seen == set(BUDGETS), f"kernels not found in the library: {set(BUDGETS) - seen}"


def _model_convs():
    """(name, B, C, H, W, K, R, stride, pad, groups) of every conv of the bench models (harness/models.py)"""
    out = []
    B = 256
    gc = [("gc1x1g2", 256, 32, 256, 1, 1, 0, 2), ("gc3x3g16", 256, 16, 512, 3, 1, 1, 16), ("gc1x1g4", 512, 16, 512, 1, 1, 0, 4),
          ("gc3x3g32", 512, 8, 1024, 3, 1, 1, 32), ("gc1x1g8", 1024, 8, 1024, 1, 1, 0, 8), ("gc_head", 1024, 8, 10, 1, 1, 0, 1)]
    nin = [("nin1x1a", 192, 32, 160, 1, 1, 0, 1), ("nin1x1b", 160, 32, 96, 1, 1, 0, 1), ("nin5x5", 96, 16, 192, 5, 1, 2, 1),
           ("nin1x1c", 192, 16, 192, 1, 1, 0, 1), ("nin3x3", 192, 8, 192, 3, 1, 1, 1), ("nin1x1d", 192, 8, 192, 1, 1, 0, 1),
           ("nin_head", 192, 8, 10, 1, 1, 0, 1)]
    for n, c, h, k, r, st, p, g in gc + nin:
        out.append((n, B, c, h, h, k, r, st, p, g))
    for hw, b, tag in ((32, 256, "res32"), (224, 64, "res224")):
        c, h = 64, hw
        out.append((f"{tag}_stem", b, 3, h, h, 64, 3, 1, 1, 1))
        for width in (64, 128, 256, 512):
            if width != 64:
                out.append((f"{tag}_{width}_s2", b, c, h, h, width, 3, 2, 1, 1))
                out.append((f"{tag}_{width}_sc", b, c, h, h, width, 1, 2, 0, 1))
                h //= 2
            out.append((f"{tag}_{width}", b, width, h, h, width, 3, 1, 1, 1))
            c = width
    return out


@pytest.mark.parametrize("conv", _model_convs(), ids=lambda c: c[0])
def test_packed_operand_plan_covers_the_bench_models(conv):
    from micronet_b200 import _lib as L
    lib = L.load()
    name, B, Cc, H, W, K, R, st, pad, G = conv
    sh = L.ConvShape(B, Cc, H, W, K, R, R, st, st, pad, pad, 1, 1, G)
    names = "Nt ntiles MT CC chunks nstage smem tmem TH TB BW n_mtiles n_items ny".split()
    Tb = min(L.PK_TERMS, L.PK_TERMS_BWD)
    cases = [(0, 1, 1), (1, Tb, 1)]                                  # quantized forward / data gradient with integer weights
    if "res" in name:
        cases += [(0, L.PK_TERMS, L.PK_TERMS), (1, Tb, Tb)]         # the fp32 x fp32 statistics conv of QuantBNFuseConv2d
    for mode, ta, tw in cases:
        plan = (C.c_int32 * 16)()
        assert lib.mnb_pk_conv_plan(C.byref(sh), mode, ta, tw, plan) == 0, (name, mode, ta, tw, lib.mnb_last_error())
        p = dict(zip(names, list(plan)[2:]))
        assert 0 < p["smem"] <= _budget("mnb_pk.cu", "kSmemBudget"), (name, p)
        assert p["tmem"] in (32, 64, 128, 256, 512) and 2 * p["MT"] * p["Nt"] <= p["tmem"], (name, p)
        assert p["nstage"] in (2, 4, 8) and p["Nt"] % 16 == 0 and p["Nt"] <= 256 and p["CC"] % 16 == 0, (name, p)
        assert 1 <= p["n_items"] < (1 << 22) and p["n_mtiles"] < (1 << 22), (name, p)           # FastDiv's exact range
        assert p["ny"] == (4 if (mode == 1 and st == 2) else 1), (name, p)                         # stride-2 data gradient: 4 phases
        assert int(lib.mnb_pk_wimage_bytes(C.byref(sh), mode, ta, tw)) >= 16
    P, Q = (H + 2 * pad - R) // st + 1, (W + 2 * pad - R) // st + 1
    if not name.startswith("res224"):            # configs[4] is inference only: no weight gradient at 224 x 224
        assert int(lib.mnb_pk_wgrad_scratch_bytes(C.byref(sh), Tb, 1)) >= 0, name
    # plane sizes: one 16-byte vector per pixel and channel octet and piece
    assert int(lib.mnb_pk_act_bytes(B, Cc, H, W, 1)) == B * ((Cc + 7) // 8) * H * W * 16
    assert int(lib.mnb_pk_act_bytes(B, K, P, Q, Tb)) == Tb * B * ((K + 7) // 8) * P * Q * 16


# B, C, H, W, K, R, groups (stride 1, 'same' padding): grouped NIN-GC layers, odd batch, 4x4 and 12x12 images, 5x5 filters
STRIDE1_SHAPES = [
    (4, 256, 32, 32, 256, 1, 2), (4, 256, 16, 16, 512, 3, 16), (4, 512, 16, 16, 512, 1, 4), (4, 512, 8, 8, 1024, 3, 32),
    (5, 1024, 8, 8, 1024, 1, 8), (3, 192, 32, 32, 160, 1, 1), (2, 64, 32, 32, 64, 3, 1), (2, 32, 16, 16, 32, 5, 1),
    (3, 48, 4, 4, 64, 1, 1), (2, 16, 12, 12, 16, 3, 1),
]
STRIDE1_CONVS = [("x".join(map(str, s)), s[0], s[1], s[2], s[3], s[4], s[5], 1, s[5] // 2, s[6]) for s in STRIDE1_SHAPES]
STRIDE1_CONVS += [c for c in _model_convs() if c[7] == 1]


@pytest.mark.parametrize("conv", STRIDE1_CONVS, ids=lambda c: c[0])
def test_packed_operand_plan_covers_pm1_and_fp32_inputs(conv):
    """forward with a +-1 (one piece), raw fp32 (PK_TERMS pieces) or asymmetric-IAO (two pieces) input against integer
    weights, data gradient and weight gradient with the backward's pieces of dy and of the saved input"""
    from micronet_b200 import _lib as L
    lib = L.load()
    name, B, Cc, H, W, K, R, st, pad, G = conv
    sh = L.ConvShape(B, Cc, H, W, K, R, R, st, st, pad, pad, 1, 1, G)
    Tb = min(L.PK_TERMS, L.PK_TERMS_BWD)
    for mode, ta, tw in [(0, 1, 1), (0, 3, 1), (0, 2, 1), (1, Tb, 1)]:
        assert lib.mnb_pk_conv_plan(C.byref(sh), mode, ta, tw, None) == 0, (name, mode, ta, tw, lib.mnb_last_error())
    for tx in (1, Tb) if not name.startswith("res224") else ():   # configs[4] is inference only: no weight gradient at 224
        assert int(lib.mnb_pk_wgrad_scratch_bytes(C.byref(sh), Tb, tx)) >= 0, (name, tx)
