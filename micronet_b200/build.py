"""Build the sm_100a shared library in-tree with nvcc (no torch involvement).

    python -m micronet_b200.build            # builds micronet_b200/lib/libmicronet_b200.so

The .so is git-ignored but travels to the GPU box with the gpurun snapshot."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libmicronet_b200.so")
SOURCES = ["mnb_quant.cu", "mnb_fused.cu", "mnb_conv_generic.cu", "mnb_conv_tc.cu", "mnb_conv_fp32_tc.cu", "mnb_conv_packed.cu", "mnb_pk.cu", "mnb_xnor.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-cudart", "static", "--expt-relaxed-constexpr",
]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "micronet_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    objs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", path, "-o", obj] + (["-Xptxas", "-v"] if verbose else [])
        subprocess.run(cmd, check=True)
        objs.append(obj)
    subprocess.run([NVCC, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-o", LIB_PATH, *objs], check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
