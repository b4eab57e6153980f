"""oracle/_ref: the reference's OWN elementwise CUDA kernels, compiled from the sources where they lie under /root/reference (nothing
is copied into this repository): activation.cu, norm.cu, rope.cu, reshape_paged_cache.cu, fp8_quant.cu, fused_qknorm_rope.cu,
moe/moe_fused_topk.cu, llm_decode_metadata_update.cu and fp8_scaled_quantize.cpp of xllm/core/kernels/cuda, with nvcc for sm_100a against the libtorch of this image.  They need no part of the reference's build system;
the only missing header is <glog/logging.h>, for which oracle/ref_stubs/ forwards to c10's glog-compatible macros.  (Attention =
FlashInfer and the FP8 GEMM = CUTLASS are un-vendored third-party code and stay "unbuildable": DESIGN.md section 2.)

Outputs only into oracle/_ref/ (git-ignored, shipped to the GPU box): libxllm_ref_kernels.so + the test binding
xllm_ref_kernels_py.so (oracle/ref_binding.cpp).  TEST INFRASTRUCTURE: tests/golden/make_ref_kernel_golden.py runs them on a GPU
and stores their outputs for tests/test_gpu_zzz_ref_kernels.py.  Needs the reference's sources.
  python -m oracle.build_ref [-f]"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
KDIR = os.path.join(REF, "xllm", "core", "kernels", "cuda")
OUT = os.path.join(HERE, "_ref")
LIB = os.path.join(OUT, "libxllm_ref_kernels.so")
PYMOD = os.path.join(OUT, "xllm_ref_kernels_py.so")
SOURCES = ["activation.cu", "norm.cu", "rope.cu", "reshape_paged_cache.cu", "fp8_quant.cu", "fused_qknorm_rope.cu",
           "moe/moe_fused_topk.cu", "llm_decode_metadata_update.cu", "fp8_scaled_quantize.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def available() -> bool:
    return os.path.exists(LIB) and os.path.exists(PYMOD)


def build(verbose=False, force=False):
    """-> path of the python module, or None when neither the reference tree nor a prebuilt oracle/_ref is present"""
    if not os.path.isdir(KDIR):
        return PYMOD if available() else None       # GPU box: no reference tree - the prebuilt files are all there is
    if available() and not force and os.path.getmtime(PYMOD) >= os.path.getmtime(os.path.join(HERE, "ref_binding.cpp")):
        return PYMOD
    import pybind11
    import sysconfig
    import torch
    import tvm_ffi
    ti = os.path.dirname(torch.__file__)
    tv = os.path.join(os.path.dirname(tvm_ffi.__file__), "include")
    os.makedirs(os.path.join(OUT, "obj"), exist_ok=True)
    inc = [f"-I{os.path.join(HERE, 'ref_stubs')}", f"-I{KDIR}", f"-I{os.path.join(KDIR, 'moe')}", f"-I{os.path.join(REF, 'xllm', 'core')}",
           f"-I{os.path.join(REF, 'xllm')}", f"-I{REF}", f"-I{ti}/include",
           f"-I{ti}/include/torch/csrc/api/include", f"-I{tv}", f"-I{sysconfig.get_paths()['include']}",      # fp8_quant.cu pulls torch/extension.h -> Python.h
           "-D_GLIBCXX_USE_CXX11_ABI=1", "-DUSE_CUDA"]
    jobs, objs = [], []
    for s in SOURCES:
        obj = os.path.join(OUT, "obj", os.path.basename(s).rsplit(".", 1)[0] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj):
            jobs.append([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "--expt-relaxed-constexpr",
                         "--expt-extended-lambda", "-Xcompiler", "-fPIC", "-w"] + inc + ["-c", os.path.join(KDIR, s), "-o", obj])

    def run(cmd):
        return cmd, subprocess.run(cmd, capture_output=True, text=True)
    with ThreadPoolExecutor(max_workers=max(1, min(6, len(jobs)))) as ex:
        for cmd, r in ex.map(run, jobs):
            if verbose or r.returncode != 0:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout[-4000:] + r.stderr[-4000:])
            if r.returncode != 0:
                raise RuntimeError("reference kernel failed to compile: " + cmd[-3])
    link = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs + \
           [f"-L{ti}/lib", "-ltorch", "-ltorch_cpu", "-ltorch_cuda", "-lc10", "-lc10_cuda", f"-Xlinker=-rpath,{ti}/lib"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("reference kernel library failed to link")
    cmd = ["g++", "-std=c++17", "-O1", "-fPIC", "-shared", os.path.join(HERE, "ref_binding.cpp"), "-o", PYMOD, f"-I{ti}/include",
           f"-I{ti}/include/torch/csrc/api/include", "-I/usr/local/cuda/include", f"-I{pybind11.get_include()}",
           f"-I{sysconfig.get_paths()['include']}", "-D_GLIBCXX_USE_CXX11_ABI=1", "-DTORCH_EXTENSION_NAME=xllm_ref_kernels_py",
           f"-L{OUT}", "-lxllm_ref_kernels", f"-L{ti}/lib", "-ltorch", "-ltorch_cpu", "-ltorch_python", "-lc10",
           f"-Wl,-rpath,{ti}/lib", "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("reference kernel binding failed to build")
    return PYMOD


def load():
    """import the binding of the reference's kernels (None when oracle/_ref is absent and cannot be built here)"""
    import importlib.util
    import torch  # noqa: F401
    so = build()
    if so is None:
        return None
    spec = importlib.util.spec_from_file_location("xllm_ref_kernels_py", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
