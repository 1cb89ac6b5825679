"""In-tree build of libguidedattn.so for sm_100a (nvcc cross-compiles without a GPU).  `python -m guided_attention_b200.build`."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
OUT = os.path.join(CSRC, "libguidedattn.so")
SOURCES = ["c_api.cu", "cross_attn_simt.cu", "cross_attn_tc.cu", "self_attn_tc.cu", "guidance_tail.cu", "step_driver.cu", "unet_ops.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-shared"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.isfile(OUT):
        return True
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    deps += [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    return any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-I", CSRC, *[os.path.join(CSRC, s) for s in SOURCES], "-o", OUT]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
