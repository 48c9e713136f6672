#!/usr/bin/env python
"""Build a variant of libstar_sm100.so with extra -D macros (the instrumented trace builds documented in the kernels'
headers), e.g.   python tools/build_variant.py gtrace -DSTAR_GEMM_TRACE=1
The variant lands in tools/variants/libstar_<tag>.so (git-ignored, travels to the GPU box); tools/kbench.py --lib <path>
and bench.py --lib <path> load it instead of the shipped library.  The product has no run-time kernel dispatch."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import CSRC, NVCC_FLAGS  # noqa: E402


def main():
    tag, defs = sys.argv[1], sys.argv[2:]
    out_dir = os.path.join(ROOT, "tools", "variants")
    os.makedirs(out_dir, exist_ok=True)
    out = os.path.join(out_dir, f"libstar_{tag}.so")
    cmd = [os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")] + NVCC_FLAGS + defs + ["-o", out, os.path.join(CSRC, "star_abi.cu")]
    subprocess.run(cmd, check=True, cwd=ROOT)
    print(out)


if __name__ == "__main__":
    main()
