"""The seeded cases on which this library's elementwise kernels are held to the reference's OWN CUDA kernels (activation.cu, norm.cu,
rope.cu, reshape_paged_cache.cu, fp8_quant.cu, fused_qknorm_rope.cu, moe/moe_fused_topk.cu, llm_decode_metadata_update.cu and
fp8_scaled_quantize.cpp of xllm/core/kernels/cuda).

tests/golden/make_ref_kernel_golden.py ran these cases through the reference's kernels (built into oracle/_ref by oracle/build_ref.py)
and stored what they computed in tests/golden/ref_kernels.pt.gz; tests/test_gpu_zzz_ref_kernels.py runs the same cases through this
library and compares.  The digest of each case's inputs is stored beside its outputs."""
import gzip
import hashlib
import io

import torch

BF16, E4M3, I32 = torch.bfloat16, torch.float8_e4m3fn, torch.int32
META_SRC = ("tokens", "positions", "new_cache_slots", "kv_seq_lens", "paged_kv_indptr", "paged_kv_indices", "paged_kv_last_page_len")
META_DST = ("tokens", "positions", "new_cache_slots", "kv_seq_lens", "kv_seq_lens_delta", "paged_kv_indptr", "paged_kv_indices",
            "paged_kv_last_page_len")
FULL_NUMEL = 1024          # outputs up to this size are stored whole; of larger ones, SAMPLE evenly spaced values
SAMPLE = 32


def tensor_bytes(t):
    t = t.detach().contiguous().cpu()
    return t.reshape(-1).view(torch.uint8).numpy().tobytes()


def cases(k, dev="cuda"):
    """-> [(case name, run)].  run() -> (digest of the case's inputs, [(op, output tensor), ...]).  `k` is this library's ops module
    or anything with the same signatures (the golden recorder adapts the reference's binding to them).

    The inputs are drawn here, up front, from one CUDA generator seeded 2026, in the order and with the expressions the live
    comparison with the reference's kernels always used, so the stored outputs are those of the same comparison.  A case never
    modifies its inputs (in-place kernels get clones): cases that share inputs see them unchanged."""
    g = torch.Generator(device=dev).manual_seed(2026)
    out = []

    def rnd(*shape, scale=1.0):
        return (torch.randn(*shape, generator=g, device=dev) * scale).to(BF16)

    def add(name, inputs, fn):
        h = hashlib.sha256()
        for t in inputs:
            h.update(tensor_bytes(t))
        digest = h.hexdigest()

        def run():
            outs = fn()
            torch.cuda.synchronize()
            return digest, outs
        out.append((name, run))

    for T, H in ((7, 3584), (64, 4096), (1, 256), (33, 1024), (300, 8192)):
        x, r0, w = rnd(T, H), rnd(T, H), (1 + 0.1 * torch.randn(H, generator=g, device=dev)).to(BF16)
        s = torch.tensor([0.05], device=dev)

        def norm(x=x, w=w):
            a = torch.empty_like(x)
            k.rms_norm(a, x, w, 1e-6)
            return [("rms_norm", a)]

        def add_norm(x=x, r0=r0, w=w):
            x1, r1 = x.clone(), r0.clone()
            k.fused_add_rms_norm(x1, r1, w, 1e-6)
            return [("fused_add_rms_norm", x1), ("fused_add_rms_norm", r1)]

        def norm_q(x=x, w=w, s=s, T=T, H=H):
            q = torch.empty(T, H, dtype=E4M3, device=dev)
            k.rms_norm_static_fp8_quant(q, x, w, s, 1e-6)
            return [("rms_norm_static_fp8_quant", q)]

        def add_norm_q(x=x, r0=r0, w=w, s=s, T=T, H=H):
            q = torch.empty(T, H, dtype=E4M3, device=dev)
            x1, r1 = x.clone(), r0.clone()
            k.fused_add_rms_norm_static_fp8_quant(q, x1, r1, w, s, 1e-6)
            return [("fused_add_rms_norm_static_fp8_quant", q), ("fused_add_rms_norm_static_fp8_quant", r1)]
        add(f"rms_norm {T}x{H}", (x, w), norm)
        add(f"fused_add_rms_norm {T}x{H}", (x, r0, w), add_norm)
        add(f"rms_norm_static_fp8_quant {T}x{H}", (x, w), norm_q)
        add(f"fused_add_rms_norm_static_fp8_quant {T}x{H}", (x, r0, w), add_norm_q)
        big = rnd(T, H, scale=5.0)
        big[0, 0] = 3000.0                                                  # saturates
        for sv in (0.5, 0.02):
            def quant(big=big, sv=sv, T=T, H=H):
                q = torch.empty(T, H, dtype=E4M3, device=dev)
                k.static_scaled_fp8_quant(q, big, torch.tensor([sv], device=dev))
                return [("static_scaled_fp8_quant", q)]
            add(f"static_scaled_fp8_quant {T}x{H} scale {sv}", (big,), quant)

    for T, d in ((7, 18944), (4 * 7, 64), (28, 129), (33, 1024)):
        gu = rnd(T, 2 * d, scale=0.5)
        for mode in ("silu", "gelu", "gelu_tanh"):
            def act(gu=gu, mode=mode, T=T, d=d):
                o = torch.empty(T, d, dtype=BF16, device=dev)
                k.act_and_mul(o, gu, mode)
                return [("act_and_mul", o)]
            add(f"act_and_mul {T}x{d} {mode}", (gu,), act)

    from xllm_b200.qwen2 import Qwen2Config, make_cos_sin_cache
    for T, HQ, HKV, D, neox in ((6, 8, 2, 16, True), (5, 6, 2, 8, False), (33, 28, 4, 128, True), (128, 32, 8, 64, True),
                                (1, 64, 8, 128, True), (7, 8, 2, 64, False)):
        cfg = Qwen2Config(hidden_size=HQ * D, num_layers=1, n_heads=HQ, n_kv_heads=HKV, head_dim=D, intermediate_size=64, vocab_size=64,
                          max_position_embeddings=max(64, T + 8), block_size=16, quant="bf16", name="rope")
        cache = make_cos_sin_cache(cfg, dev)
        pos = torch.tensor([(i * 3 + 1) % cache.size(0) for i in range(T)], dtype=torch.int64, device=dev)
        q, kk = rnd(T, HQ * D), rnd(T, HKV * D)

        def rope(pos=pos, q=q, kk=kk, cache=cache, neox=neox):
            q1, k1 = q.clone(), kk.clone()
            k.rotary_embedding(pos, q1, k1, cache, neox)
            return [("rotary_embedding", q1), ("rotary_embedding", k1)]
        add(f"rotary_embedding T{T} {HQ}/{HKV}x{D} neox={neox}", (pos, q, kk, cache), rope)

    for n_tokens, n_blocks, bs, hkv, D in ((4, 1, 16, 1, 64), (32, 8, 16, 4, 128), (64, 4, 64, 8, 128), (256, 16, 64, 8, 128),
                                           (1, 4, 16, 4, 128)):
        keys, vals = rnd(n_tokens, hkv, D), rnd(n_tokens, hkv, D)
        slots = torch.randperm(n_blocks * bs, generator=g, device=dev)[:n_tokens].to(I32)

        def scatter(keys=keys, vals=vals, slots=slots, shape=(n_blocks, bs, hkv, D)):
            kc = torch.zeros(*shape, dtype=BF16, device=dev)
            vc = torch.zeros_like(kc)
            k.reshape_paged_cache(slots, keys, vals, kc, vc)
            return [("reshape_paged_cache", kc), ("reshape_paged_cache", vc)]
        add(f"reshape_paged_cache {n_tokens} tokens {n_blocks}x{bs} blocks {hkv}x{D}", (keys, vals, slots), scatter)

    for T, hq, hk, D, maxpos, inter in ((17, 8, 4, 128, 512, False), (11, 6, 2, 64, 256, True), (3, 16, 2, 128, 64, False)):
        qkv = rnd(T, (hq + 2 * hk) * D, scale=0.2)
        qw, kw = rnd(D), rnd(D)
        cache = torch.randn(maxpos, D, generator=g, device=dev).to(BF16)
        pos = torch.randint(0, maxpos, (T,), generator=g, device=dev)

        def qknorm(qkv=qkv, qw=qw, kw=kw, cache=cache, pos=pos, hq=hq, hk=hk, D=D, inter=inter):
            a = qkv.clone()
            k.fused_qk_norm_rope(a, hq, hk, hk, D, 1e-6, qw, kw, cache, inter, pos)
            return [("fused_qk_norm_rope", a)]
        add(f"fused_qk_norm_rope T{T} {hq}/{hk}x{D} interleaved={inter}", (qkv, qw, kw, cache, pos), qknorm)

    # dynamic per-tensor FP8 quantisation (fp8_scaled_quantize.cpp:36-41: the scale is formed in the tensor's dtype, then cast)
    for T, H, sc in ((7, 3584, 1.0), (32, 8192, 5.0), (1, 256, 0.01), (64, 1024, 40.0)):
        x = rnd(T, H, scale=sc)

        def dyn(x=x):
            q, s = k.fp8_scaled_quantize(x)
            return [("fp8_scaled_quantize", q), ("fp8_scaled_quantize", s.reshape(-1).float())]
        add(f"fp8_scaled_quantize {T}x{H} x{sc}", (x,), dyn)

    # MoE router: expert ids are index work (held to identity); the fp32 routing weights to 1e-6 relative
    for T, E, topk, dt in ((7, 16, 2, torch.float32), (33, 64, 8, torch.float32), (512, 16, 2, BF16), (5, 256, 8, BF16),
                           (1, 8, 1, torch.float32)):
        logits = (torch.randn(T, E, generator=g, device=dev) * 3).to(dt)
        bias = torch.randn(E, generator=g, device=dev) * 0.1
        for scoring, use_bias in (("softmax", False), ("sigmoid", False), ("sigmoid", True)):
            for renorm in (True, False):
                def router(logits=logits, bias=bias if use_bias else None, topk=topk, renorm=renorm, scoring=scoring):
                    w, ids = k.moe_fused_topk(logits.clone(), topk, renorm, bias, scoring)
                    return [("moe_fused_topk_ids", ids.to(I32)), ("moe_fused_topk_weights", w.float())]
                add(f"moe_fused_topk {T}x{E} top{topk} {str(dt).split('.')[-1]} {scoring} bias={use_bias} renorm={renorm}",
                    (logits, bias), router)

    # CUDA-graph decode metadata refresh: integer work, every destination buffer compared whole
    for n_tok, padded, batch, n_idx in ((5, 8, 5, 37), (1, 1, 1, 1), (64, 64, 64, 4000), (3, 16, 3, 0), (300, 512, 300, 70000)):
        ri = lambda n, hi=100000: torch.randint(0, hi, (n,), generator=g, device=dev, dtype=I32)   # noqa: E731
        zero = torch.zeros(1, dtype=I32, device=dev)
        src = dict(tokens=ri(n_tok), positions=ri(n_tok), new_cache_slots=ri(n_tok),
                   kv_seq_lens=torch.cat([zero, ri(batch, 500).cumsum(0).to(I32)]),
                   paged_kv_indptr=torch.cat([zero, ri(batch, 40).cumsum(0).to(I32)]), paged_kv_indices=ri(max(n_idx, 1)),
                   paged_kv_last_page_len=ri(max(batch, 1), 128) + 1)
        cap_tok, cap_batch, cap_idx = max(padded, n_tok) + 7, batch + 5, n_idx + 11
        dst = dict(tokens=ri(cap_tok), positions=ri(cap_tok), new_cache_slots=ri(cap_tok), kv_seq_lens=ri(cap_batch + 1),
                   kv_seq_lens_delta=ri(cap_batch), paged_kv_indptr=ri(cap_batch + 1), paged_kv_indices=ri(cap_idx),
                   paged_kv_last_page_len=ri(cap_batch))

        def metadata(src=src, dst=dst, args=(n_tok, padded, batch, n_idx)):
            d = {f: t.clone() for f, t in dst.items()}
            k.update_llm_decode_metadata(src, d, *args)
            return [("update_llm_decode_metadata", d[f]) for f in META_DST]
        add(f"update_llm_decode_metadata tokens {n_tok}/{padded} batch {batch} indices {n_idx}",
            [src[f] for f in META_SRC] + [dst[f] for f in META_DST], metadata)
    return out


def stored_values(t):
    """the values of an output that the golden file keeps, in the output's own dtype: all of them when few, else SAMPLE evenly
    spaced ones"""
    flat = t.detach().reshape(-1).cpu()
    if flat.numel() <= FULL_NUMEL:
        return flat.clone()
    return flat[torch.linspace(0, flat.numel() - 1, SAMPLE).long()]


def record(t):
    """what the golden file keeps of one output: dtype, shape, a digest of its bytes and stored_values()"""
    return {"dtype": str(t.dtype), "shape": list(t.shape), "sha256": hashlib.sha256(tensor_bytes(t)).hexdigest(),
            "values": stored_values(t)}


def save_golden(obj, path):
    buf = io.BytesIO()
    torch.save(obj, buf)
    with open(path, "wb") as f:
        f.write(gzip.compress(buf.getvalue(), 9, mtime=0))


def load_golden(path):
    with open(path, "rb") as f:
        return torch.load(io.BytesIO(gzip.decompress(f.read())), weights_only=True)
