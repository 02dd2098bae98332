"""TEST INFRASTRUCTURE (oracle) -- builds the UNMODIFIED reference segment tree.

Compiles the reference's own C++/CUDA segment-tree sources *where they lie* under
$RLB_REFERENCE_ROOT/torchrl/csrc (a torchrl source checkout; nothing is copied into this repo) into

    oracle/_ref/cpu/_torchrl.so    SumSegmentTreeFp32/64, MinSegmentTreeFp32/64   (csrc/pybind.cpp:21-38)
    oracle/_ref/cuda/_torchrl.so   ... plus CudaSum/MinSegmentTreeFp32/64          (csrc/cuda_segment_tree.cu)

The outputs are git-ignored.  They serve (a) to record the reference tapes the parity tests play
back (tests/golden/README.md) and (b) as the "reference" arm of bench.py (cpu_baseline.kind ==
"reference").  The module name must stay ``_torchrl`` because the reference registers
PYBIND11_MODULE(_torchrl, m).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
load these files.  The product package (rl_b200) never imports anything under oracle/.
"""
from __future__ import annotations

import os
import sys
from pathlib import Path

OUT = Path(__file__).resolve().parent / "_ref"


def build(with_cuda: bool, verbose: bool = False) -> Path:
    from torch.utils.cpp_extension import load

    kind = "cuda" if with_cuda else "cpu"
    out = OUT / kind
    so = out / "_torchrl.so"
    if so.exists():
        return so
    root = os.environ.get("RLB_REFERENCE_ROOT")
    csrc = Path(root or ".") / "torchrl" / "csrc"
    if not root or not csrc.is_dir():
        raise FileNotFoundError(f"{so} is not built and RLB_REFERENCE_ROOT names no torchrl source checkout")
    out.mkdir(parents=True, exist_ok=True)
    sources = [str(csrc / "pybind.cpp"), str(csrc / "utils.cpp")]
    cflags = ["-O3", "-std=c++17"]
    kwargs = {}
    if with_cuda:
        # setup.py:74-92 would skip CUDA on an nvcc/torch minor mismatch unless FORCE_CUDA=1; force it.
        sources.append(str(csrc / "cuda_segment_tree.cu"))
        cflags.append("-DWITH_CUDA")
        os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
        kwargs.update(with_cuda=True, extra_cuda_cflags=["-O3", "-std=c++17", "-DWITH_CUDA"])
    load(name="_torchrl", sources=sources, extra_cflags=cflags, build_directory=str(out),
         verbose=verbose, is_python_module=False, **kwargs)
    assert so.exists(), so
    return so


if __name__ == "__main__":
    kinds = sys.argv[1:] or ["cpu", "cuda"]
    for k in kinds:
        print(build(with_cuda=(k == "cuda"), verbose=True))
