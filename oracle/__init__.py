"""CPU oracle for the xLLM per-layer inference hot path.  TEST INFRASTRUCTURE ONLY.

This package restates, op by op, the arithmetic of the reference
(jd-opensource/xllm @ 87e8d6e, v0.9.0) for the path named in BASELINE.json:
paged attention, the (quantised) linears, RMSNorm, RoPE, SiLU*mul, the KV-cache
scatter and the integer page-table metadata.  Every function cites the
reference file:line it follows (paths relative to the reference checkout).

Who may import it: tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs, as the CHECKER or as the timed CPU baseline.  The product
(xllm_b200/) never imports it and has no CPU fallback.

Parity pinning (SURVEY.md 8c):
  * integer page-table metadata  -> pinned by BatchTest.Basic golden vectors
    (tests/core/framework/batch/batch_test.cpp:403-546), tests/test_oracle_golden.py
  * attention layer composition (qkv+bias -> rope -> paged attention -> o_proj)
    -> pinned by the known answers of tests/core/layers/mlu/qwen2_attention_test.cpp:254-393
    with the seeded_tensor generator (tests_utils.cpp:159-274); values produced on
    MLU hardware, reproduced here to bf16 rounding (see the test for the tolerance)
  * RMSNorm / RoPE / KV scatter / SiLU*mul / FP8 quant follow the reference .cu
    files line by line; the reference's own kernel tests (torch expressions, no
    stored vectors) are restated on the oracle in tests/test_oracle_reference_kats_cpu.py,
    and the reference's kernels THEMSELVES are compiled from its sources into
    oracle/_ref/ (oracle/build_ref.py); their outputs on the cases of
    tests/ref_kernel_cases.py are stored in tests/golden/ref_kernels.pt.gz, which
    tests/test_gpu_zzz_ref_kernels.py compares the CUDA kernels with
  * MoE router -> pinned by the known answers of tests/core/layers/mlu/moe_gate_test.cpp:143-268
    (tests/test_moe_cpu.py); whole-model composition -> transformers' Qwen2 / Llama
    (tests/test_oracle_vs_transformers_cpu.py)
  * CUDA paged-attention numerics live in un-vendored FlashInfer v0.6.2
    (docker/Dockerfile.cuda:16): restated from its published algorithm
    (fp32 scores, base-2 online softmax, P rounded to bf16, denominator summed
    from the rounded P, fp32 accumulate) - "parity unpinned" by any reference test
  * W4A16 / W8A16 linears do not exist in the reference: the oracle DEFINES the
    spec (oracle/quant.py) - "parity unpinned"
The reference C++ cannot be compiled here (needs glog/gflags/folly/brpc/boost,
13 empty submodules, and has no CPU build: xllm/models/models.h:119-121), so there
is no oracle/_ref.
"""
