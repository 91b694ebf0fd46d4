"""Hardware self-tests of the sm_100a building blocks (tcgen05 descriptors, TMA geometry)."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _err_flag():
    return torch.zeros(1, dtype=torch.int32, device=DEV)


@pytest.mark.parametrize("int8", [0, 1, 2])  # 0: bf16 K-major, 1: int8 K-major, 2: bf16 MN-major operands
@pytest.mark.parametrize("N,K", [(16, 32), (32, 64), (64, 32), (128, 64), (48, 64)])
def test_umma_descriptor_selftest(N, K, int8):
    from micronet_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(N * 1000 + K + int8)
    lo, hi = (-128, 128) if int8 == 1 else (-16, 17)
    A = torch.randint(lo, hi, (128, K), generator=g).float()
    B = torch.randint(lo, hi, (N, K), generator=g).float()
    want = A.double() @ B.double().t()
    Ad, Bd = A.to(DEV), B.to(DEV)
    D = torch.full((128, N), float("nan"), device=DEV)
    err = _err_flag()
    L.check(lib.mnb_selftest_umma(Ad.data_ptr(), Bd.data_ptr(), D.data_ptr(), N, K, int8, err.data_ptr(),
                                  L.stream()), "selftest_umma")
    torch.cuda.synchronize()
    assert err.item() == 0, f"bounded wait timed out (code {err.item()})"
    assert torch.equal(D.cpu().double(), want), (D.cpu()[:2, :8], want[:2, :8])


TMA_CASE = r"""
import ctypes as C, sys, torch
sys.path.insert(0, sys.argv[1])
from micronet_b200 import _lib as L
coord = tuple(int(v) for v in sys.argv[2:5])
lib = L.load()
Wd, Hd, Cd = 20, 10, 6
box = (8, 4, 2)
src = torch.arange(Wd * Hd * Cd, dtype=torch.float32).reshape(Cd, Hd, Wd) + 1.0
pad = torch.zeros(Cd + 8, Hd + 16, Wd + 32)
pad[:Cd, 8:8 + Hd, 16:16 + Wd] = src
pad = torch.nn.functional.pad(pad, (0, 0, 0, 0, 4, 0))  # room for negative channel coordinates
want = pad[4 + coord[2]:4 + coord[2] + box[2], 8 + coord[1]:8 + coord[1] + box[1], 16 + coord[0]:16 + coord[0] + box[0]]
out = torch.full((box[2], box[1], box[0]), float("nan"), device="cuda:0")
err = torch.zeros(1, dtype=torch.int32, device="cuda:0")
sd = src.to("cuda:0")
L.check(lib.mnb_selftest_tma3d(sd.data_ptr(), (C.c_int64 * 3)(Wd, Hd, Cd), (C.c_int32 * 3)(*box),
                               (C.c_int32 * 3)(*coord), out.data_ptr(), err.data_ptr(), L.stream()), "selftest_tma3d")
torch.cuda.synchronize()
assert err.item() == 0, f"bounded wait timed out (code {err.item()})"
assert torch.equal(out.cpu(), want), (out.cpu(), want)
print("TMA_OK")
"""

# inner coordinate must stay 16-byte aligned (multiples of 4 floats); outer coordinates may be
# negative / past the end and read back as zeros.  One process per case: a faulting TMA poisons
# the CUDA context.
TMA_COORDS = [(0, 0, 0), (4, -1, 0), (16, 8, 4), (12, -3, 5), (-4, 7, 1), (8, 9, -1)]


@pytest.mark.parametrize("coord", TMA_COORDS, ids=[str(c) for c in TMA_COORDS])
def test_tma_box_and_oob_fill(coord, tmp_path):
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "tma_case.py"
    script.write_text(TMA_CASE)
    out = subprocess.run([sys.executable, str(script), root, *map(str, coord)], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0 and "TMA_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
