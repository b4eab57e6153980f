"""Runs the cases of tests/ref_kernel_cases.py through the REFERENCE'S OWN CUDA kernels and stores what they computed as
tests/golden/ref_kernels.pt.gz, which tests/test_gpu_zzz_ref_kernels.py holds this library's kernels to.

Needs a GPU and the reference's kernels compiled into oracle/_ref (python -m oracle.build_ref, on a machine with the reference's
sources); nothing else in the repository needs either.

    python tests/golden/make_ref_kernel_golden.py [out.pt.gz]        # default: rewrites tests/golden/ref_kernels.pt.gz (commit the result)
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import build_ref                                  # noqa: E402
from tests.ref_kernel_cases import META_DST, META_SRC, cases, record, save_golden   # noqa: E402


class ReferenceAsLibrary:
    """the reference's binding (oracle/ref_binding.cpp) behind this library's ops signatures"""

    def __init__(self, ref):
        self.ref = ref

    def __getattr__(self, name):
        return getattr(self.ref, name)

    def fp8_scaled_quantize(self, x):
        return self.ref.fp8_scaled_quantize(x, None, None)

    def update_llm_decode_metadata(self, src, dst, n_tok, padded, batch, n_idx):
        self.ref.update_llm_decode_metadata([src[f] for f in META_SRC], [dst[f] for f in META_DST], n_tok, padded, batch, n_idx)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_kernels.pt.gz")
    ref = build_ref.load()
    if ref is None:
        sys.exit("oracle/_ref is not built: python -m oracle.build_ref needs the reference's sources")
    golden = {}
    for name, run in cases(ReferenceAsLibrary(ref)):
        digest, outs = run()
        golden[name] = {"inputs_sha256": digest,
                        "outputs": [dict(op=op, **record(t)) for op, t in outs]}
    save_golden({"device": torch.cuda.get_device_name(0), "torch": str(torch.__version__), "cases": golden}, out_path)
    print(f"{len(golden)} cases -> {out_path} ({os.path.getsize(out_path)} bytes)")


if __name__ == "__main__":
    main()
