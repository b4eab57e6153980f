"""This library's elementwise kernels against what the REFERENCE'S OWN CUDA kernels computed on the same inputs: activation.cu,
norm.cu, rope.cu, reshape_paged_cache.cu, fp8_quant.cu, fused_qknorm_rope.cu, moe/moe_fused_topk.cu, llm_decode_metadata_update.cu and
fp8_scaled_quantize.cpp, run on a B200 over the seeded cases of tests/ref_kernel_cases.py by tests/golden/make_ref_kernel_golden.py and
stored in tests/golden/ref_kernels.pt.gz (per output: a digest of its bytes and its values, all or evenly spaced ones).

Per op the report counts the cases whose outputs are bit-identical to the reference's; otherwise it keeps the worst difference over
the stored values.  Every op here is also held bit-exact to the oracle's restatement of the same sources elsewhere in the suite."""
import hashlib
import os

import pytest
import torch

from tests.ref_kernel_cases import cases, load_golden, stored_values, tensor_bytes

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.pt.gz")
OPS = ["rms_norm", "fused_add_rms_norm", "rms_norm_static_fp8_quant", "fused_add_rms_norm_static_fp8_quant", "static_scaled_fp8_quant",
       "act_and_mul", "rotary_embedding", "reshape_paged_cache", "fused_qk_norm_rope", "fp8_scaled_quantize", "moe_fused_topk_ids", "update_llm_decode_metadata"]


def _compare(t, ref):
    """-> (bit identical, max abs difference over the stored values, how many of them differ, max relative difference)"""
    same = str(t.dtype) == ref["dtype"] and list(t.shape) == ref["shape"] and hashlib.sha256(tensor_bytes(t)).hexdigest() == ref["sha256"]
    a, b = stored_values(t).to(torch.float64), ref["values"].to(torch.float64)
    differ = (a != b) & ~(a.isnan() & b.isnan())
    d = torch.where(differ, (a - b).abs(), torch.zeros_like(a))
    rel = torch.where(differ, d / b.abs().clamp_min(1e-30), torch.zeros_like(a))
    return same, float(d.max()) if d.numel() else 0.0, int(differ.sum()), float(rel.max()) if rel.numel() else 0.0


@pytest.fixture(scope="module")
def parity(built_lib):
    from xllm_b200 import ops
    golden = load_golden(GOLDEN)["cases"]
    todo = cases(ops)
    assert sorted(name for name, _ in todo) == sorted(golden), "tests/ref_kernel_cases.py and tests/golden/ref_kernels.pt.gz disagree"
    res = {}

    def entry(op):
        return res.setdefault(op, {"cases": 0, "bit_identical": 0, "worst": None, "errors": []})
    for name, run in todo:
        g = golden[name]
        ref_ops = sorted({o["op"] for o in g["outputs"]})
        try:
            digest, outs = run()
        except Exception as e:                                              # noqa: BLE001
            for op in ref_ops:
                r = entry(op)
                r["cases"] += 1
                r["errors"].append(f"{name}: {type(e).__name__}: {str(e)[:160]}")
            continue
        assert digest == g["inputs_sha256"], f"{name}: the inputs differ from those the golden outputs were recorded on"
        assert [op for op, _ in outs] == [o["op"] for o in g["outputs"]], name
        for op in ref_ops:
            r = entry(op)
            r["cases"] += 1
            cmp = [_compare(t, ref) for (o, t), ref in zip(outs, g["outputs"]) if o == op]
            if all(c[0] for c in cmp):
                r["bit_identical"] += 1
            else:
                d, n = max(c[1] for c in cmp), sum(c[2] for c in cmp)
                if r["worst"] is None or d > r["worst"]["max_abs_diff"]:
                    r["worst"] = {"case": name, "max_abs_diff": d, "stored_values_differing": n}
            r["max_rel_diff"] = max(r.get("max_rel_diff", 0.0), max(c[3] for c in cmp))
    return res


# In one of their five stored cases (300 x 8192) the two fused add+RMSNorm kernels round some elements differently from the
# reference's: a parity finding against the reference, reported as XFAIL.  Every other op is bit-identical to the reference's
# kernel on every stored case and must stay so.
ROUNDING_DIFFERS = ("fused_add_rms_norm", "fused_add_rms_norm_static_fp8_quant")


@pytest.mark.parametrize("op", [pytest.param(op, marks=pytest.mark.xfail(strict=False, reason="XPASS = bit-identical to the reference's kernel"))
                                if op in ROUNDING_DIFFERS else op for op in OPS])
def test_kernel_is_bit_identical_to_the_reference_kernel(op, parity):
    r = parity[op]
    assert r["cases"] > 0 and not r.get("errors"), f"{op}: {r.get('errors')}"
    assert r["bit_identical"] == r["cases"], f"{op}: {r['bit_identical']} / {r['cases']} cases bit-identical; worst {r['worst']}"


def test_router_weights_match_the_reference_kernel(parity):
    """fp32 routing weights: the reference has two softmax kernels (fused for power-of-two expert counts, generic otherwise) whose
    reductions sum in different orders, so the floating-point bar is 1e-6 relative rather than bit identity (the expert ids - index
    work - are held to identity above)."""
    r = parity["moe_fused_topk_weights"]
    assert r["cases"] > 0 and not r.get("errors"), r.get("errors")
    assert r["bit_identical"] == r["cases"] or r.get("max_rel_diff", 1.0) <= 1e-6, r
