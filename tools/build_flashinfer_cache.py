"""Pre-builds (nvcc, no GPU needed) the FlashInfer fa2 modules that tests/test_gpu_flashinfer_pin.py and bench.py's
GPU comparators load, into baseline/_fi/ (git-ignored, travels to the GPU box with the snapshot like our own .so files).

FlashInfer is LIBRARY code here: it is the implementation the reference dlopen()s for batch_decode / batch_prefill /
batch_chunked_prefill (xllm/core/kernels/cuda/utils.cpp:371-450; reference pin v0.6.2, this image ships 0.6.11 with
the same fa2 templates).  It is used only as a checker (tests) and as a same-box comparator (bench), never on the
product path.  On a fresh GPU box the JIT would otherwise spend minutes of charged box time in nvcc per variant.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FI_BASE = os.path.join(ROOT, "baseline", "_fi")


def set_env(base=FI_BASE):
    os.environ["FLASHINFER_WORKSPACE_BASE"] = base
    os.environ["FLASHINFER_CUDA_ARCH_LIST"] = "10.0a"
    os.makedirs(base, exist_ok=True)


def specs(head_dims=(128, 64)):
    import torch
    from flashinfer.jit.attention.modules import gen_batch_decode_module, gen_batch_prefill_module
    bf, i32 = torch.bfloat16, torch.int32
    out = []
    for d in head_dims:
        out.append(gen_batch_decode_module(bf, bf, bf, i32, d, d, 0, False, False))
        out.append(gen_batch_prefill_module("fa2", bf, bf, bf, i32, d, d, 0, False, False, False))
    return out


def main():
    set_env()
    dims = tuple(int(a) for a in sys.argv[1:]) or (128, 64)
    for s in specs(dims):
        print("building", s.name, flush=True)
        s.build(verbose=False)
        print("  ->", s.jit_library_path, os.path.getsize(s.jit_library_path) >> 20, "MiB", flush=True)


if __name__ == "__main__":
    main()
