#!/usr/bin/env python
"""bench.py -- decode tokens/s of the Qwen2-7B W4A16 hot path at ctx 4096 (BASELINE.json configs[1]).

A "step" is one decode step of the whole Qwen2-7B stack (28 layers: RMSNorm, W4A16 qkv, RoPE+KV scatter, paged
decode attention over 4096 cached tokens, W4A16 o_proj, RMSNorm, W4A16 gate_up, SiLU*mul, W4A16 down; final norm,
bf16 lm_head, greedy argmax) for batch 1, replayed as one CUDA graph of libxllm_b200_ops launches.
Synthetic data: random-init weights of the named architecture, KV cache N(0,1) with a random page permutation.

  value   tokens/s with the step inputs resident in HBM (device events around K replays)
  e2e     tokens/s through Qwen2DecodeRunner.step(): pinned-host step inputs -> H2D -> graph -> D2H token ids
  roofline  dominant kernel (W4A16 gate_up_proj GEMV with the fused SiLU*mul epilogue - the variant the graph runs -
            28 launches/step): algorithmic bytes / launch duration, CUDA events around each launch in an instrumented
            pass; plus the paged decode attention kernel the north-star names, and the whole-step bytes/time
  cpu_baseline  the oracle's restatement of one decoder layer (+ lm_head) on the host cores, bounded sample,
            median of >= 5 passes with the spread reported
  comparators   same-box library kernels (NOT the reference arm): FlashInfer fa2 decode / prefill (what the reference
            dlopen()s), F.linear bf16 (cuBLASLt, the reference's matmul), torch._scaled_mm fp8 (CUTLASS stand-in)
  tp_parity (N > 1) tiny-config TP-vs-single-GPU logits / tokens / cross-rank bit-identity check, run BEFORE the timed
            region; the run exits non-zero when it fails

N > 1 (torchrun): tensor parallelism as the reference shards the path (SURVEY 8e): column-parallel qkv / gate_up / lm_head,
row-parallel o / down with one exchange after each, done by this library's NVLink one-shot all-reduce fused with the
following add+RMSNorm (NCCL all-gather for the logits).  Qwen2-7B has 28 q heads, so tp = min(N, 4); at N = 8 two TP4
groups each decode their own request (data parallel replicas of the TP4 group).  `--parallelism dp` runs N independent
replicas instead.  value = tokens of all groups / max time over ranks.
`--impl reference` times the oracle port on the host cores (the reference has no CPU build and cannot be installed
offline: see DESIGN.md) and prints the same line with "impl": "reference".
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "decode_tokens_per_s"
UNIT = "tokens/s"
CTX = 4096
WORKLOAD = "Qwen2-7B W4A16 (group 128), batch=1, ctx=4096, decode-only PagedAttention, 1xB200 per replica"


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def profiled_traffic(name):
    """DRAM bytes (read + write) per launch from a committed `ncu --set full` summary (profiles/, written by
    tools/ncu_summary.py) of the SAME kernel variant and shape.  A cross-reference, not a live measurement: the key
    `traffic_source` names the file so a stale summary is visible.  None when the summary is absent."""
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        for ln in open(os.path.join(ROOT, "profiles", name)):
            if ln.startswith("traffic = dram read + write ="):
                parts = ln.split("=")[-1].split("+")
                total = 0.0
                for part in parts:
                    v, u = part.split()
                    total += float(v) * unit[u]
                return int(total)
    except Exception:
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    """threads the CPU arm may use: the affinity mask, clipped by the cgroup CPU quota when there is one (a GPU box
    can show 128 CPUs in the mask while the container is throttled to a few), and by 32 - a batch-1 GEMV does not
    scale past that and oversubscription makes it slower."""
    n = len(os.sched_getaffinity(0))
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    return max(1, min(n, 32))


# ----------------------------------------------------------------------------------------------------------------
def cpu_layer_baseline(threads=None, budget_s=20.0):
    """The oracle port of one Qwen2-7B decoder layer (decode, batch 1, ctx 4096) + lm_head on the host cores.
    Weights are kept as fp32 copies of bf16-representable values so the timed region is the layer math, not dtype
    conversion.  Every pass is timed on its own; the MEDIAN of >= 5 passes is reported with the min..max spread (a
    shared box makes single passes noisy).  Returns (tokens/s extrapolated to 28 layers + lm_head, step seconds,
    threads, sample description, spread dict)."""
    import torch
    from oracle import layer as OL
    from oracle import ops as O
    from xllm_b200.qwen2 import Qwen2Config
    cfg = Qwen2Config.qwen2_7b()
    threads = threads or host_threads()
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(2026)
    H, I, bs = cfg.hidden_size, cfg.intermediate_size, cfg.block_size
    BF16 = torch.bfloat16

    def w(n, k):
        return (torch.randn(n, k, generator=g) * 0.02).to(BF16).to(torch.float32)   # dequantised W4 weights live as values
    qkv_w, o_w, gu_w, dn_w = w(cfg.q_size + 2 * cfg.kv_size, H), w(H, cfg.q_size), w(2 * I, H), w(H, I)
    qkv_b = (torch.randn(cfg.q_size + 2 * cfg.kv_size, generator=g) * 0.02).to(BF16)
    npg = CTX // bs
    kc = torch.randn(npg + 1, bs, cfg.n_kv_heads, cfg.head_dim, generator=g).to(BF16)
    vc = torch.randn(npg + 1, bs, cfg.n_kv_heads, cfg.head_dim, generator=g).to(BF16)
    cs = O.compute_cos_sin_cache(cfg.head_dim, 8192, cfg.rope_theta, BF16)
    lin = lambda x, ww, b=None: O.linear(x, ww, b)
    attn = OL.Qwen2AttentionOracle(qkv_w, qkv_b, o_w, cfg.n_heads, cfg.n_kv_heads, cfg.head_dim, cs, linear=lin)
    ones = torch.ones(H, dtype=BF16)
    dl = OL.Qwen2DecoderLayerOracle(attn, ones, ones, cfg.rms_norm_eps, lambda h: O.linear(h, gu_w), lambda h: O.linear(h, dn_w))
    indices = (torch.randperm(npg, generator=g) + 1).to(torch.int32)
    slot = int(indices[-1]) * bs + (CTX - 1) % bs
    meta = OL.AttnMeta(False, False, torch.tensor([0, 1], dtype=torch.int32), None, torch.tensor([slot], dtype=torch.int32),
                       torch.tensor([0, npg], dtype=torch.int32), indices, torch.tensor([(CTX - 1) % bs + 1], dtype=torch.int32))
    x = torch.randn(1, H, generator=g).to(BF16)
    res = torch.randn(1, H, generator=g).to(BF16)
    pos = torch.tensor([CTX - 1])
    dl.forward(x, res, pos, meta, kc, vc)                      # warm-up
    dl.forward(x, res, pos, meta, kc, vc)
    t_start, layer_t = time.perf_counter(), []
    while True:
        t0 = time.perf_counter()
        dl.forward(x, res, pos, meta, kc, vc)
        layer_t.append(time.perf_counter() - t0)
        if len(layer_t) >= 5 and (time.perf_counter() - t_start > budget_s * 0.7 or len(layer_t) >= 60):
            break
    head_rows = 19008                                          # 1/8 of the vocabulary rows, scaled up
    head = w(head_rows, H)
    O.linear(x, head)
    t_start, head_t = time.perf_counter(), []
    while True:
        t0 = time.perf_counter()
        O.linear(x, head)
        head_t.append(time.perf_counter() - t0)
        if len(head_t) >= 5 and (time.perf_counter() - t_start > budget_s * 0.2 or len(head_t) >= 30):
            break
    scale = cfg.vocab_size / head_rows
    t_layer, t_head = statistics.median(layer_t), statistics.median(head_t) * scale
    step_s = cfg.num_layers * t_layer + t_head
    step_fast = cfg.num_layers * min(layer_t) + min(head_t) * scale
    step_slow = cfg.num_layers * max(layer_t) + max(head_t) * scale
    sample = (f"median of {len(layer_t)} passes of one Qwen2-7B decoder layer (decode, batch 1, ctx {CTX}, dequantised "
              f"fp32-held weights) + median of {len(head_t)} passes over 1/8 of lm_head, extrapolated to {cfg.num_layers} "
              f"layers + full lm_head")
    spread = {"tokens_per_s_min": 1.0 / step_slow, "tokens_per_s_max": 1.0 / step_fast, "layer_passes": len(layer_t),
              "layer_ms_median": t_layer * 1e3, "layer_ms_min": min(layer_t) * 1e3, "layer_ms_max": max(layer_t) * 1e3}
    return 1.0 / step_s, step_s, threads, sample, spread


def run_reference(args, rank, world):
    if rank != 0:
        return
    tps, step_s, threads, sample, spread = cpu_layer_baseline(budget_s=min(60.0, 6.0 * max(1, args.steps)))
    line = {"metric": METRIC, "value": tps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "impl": "reference", "config": {"workload": WORKLOAD, "ctx": CTX, "batch": 1},
            "cpu_baseline": {"value": tps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "spread": spread},
            "e2e": {"value": tps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference has no CPU build (xllm/models/models.h:119-121 #error) and cannot be installed offline; "
                    "this arm times the oracle port of the same decoder layer on the host cores"}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
def _events_per_launch(torch, fns, reps=3):
    """CUDA events around EACH launch (first repetition dropped).  A few ms of queued GPU work first, so every launch +
    event is already enqueued when the GPU reaches it: the pairs bracket device time, not Python launch latency."""
    ev = []
    torch.cuda._sleep(int(20e6))
    for rep in range(reps):
        for fn in fns:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            if rep > 0:
                ev.append((a, b))
    torch.cuda.synchronize()
    us = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    return sum(us) / len(us), us[len(us) // 2]


def _events_chained(torch, fns, reps=5):
    """mean duration of a launch inside a back-to-back stream of launches (one per layer: different weights / caches,
    together larger than L2), events around the whole batch.  Consecutive launches are PDL-chained exactly as inside
    the decode step, so a kernel's launch latency and prologue overlap its predecessor's tail."""
    for fn in fns:
        fn()
    torch.cuda.synchronize()
    torch.cuda._sleep(int(20e6))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        for fn in fns:
            fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (reps * len(fns))


def _time_fn(torch, fn, it=5):
    fn(); fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(it):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / it * 1e-3


def gpu_comparators(torch, ops, cfg, runner, weights, dev, ctx):
    """Same-box LIBRARY kernels next to ours (extra keys; not the reference arm, never on the product path):
    FlashInfer fa2 (the module the reference dlopen()s: kernels/cuda/utils.cpp:371-450), F.linear bf16 = cuBLASLt (the
    reference's matmul, matmul.cpp:20-24), torch._scaled_mm fp8 (stand-in for cutlass_scaled_mm).  us per call."""
    out = []

    def add(name, ours_us, theirs_us, note=None):
        d = {"name": name, "ours_us": round(ours_us, 2), "theirs_us": round(theirs_us, 2),
             "speedup_vs_library": round(theirs_us / ours_us, 3)}
        if note:
            d["note"] = note
        out.append(d)
    D, HQ, HKV = cfg.head_dim, cfg.n_heads, cfg.n_kv_heads
    BF16 = torch.bfloat16
    sc = D ** -0.5
    # ---- attention: FlashInfer fa2 -------------------------------------------------------------------------------
    fi_tmp = tempfile.mkdtemp(prefix="xb_bench_flashinfer_")
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import build_flashinfer_cache as FIC
        # FlashInfer writes a log, lock files (cached_ops/tmp) and JIT output under its workspace: give it a temporary one, with
        # the modules pre-built in the tree linked in one by one
        FIC.set_env(fi_tmp)
        import flashinfer
        from flashinfer.jit import core as jc
        from flashinfer.jit import env as je
        prebuilt = os.path.join(FIC.FI_BASE, os.path.relpath(je.FLASHINFER_JIT_DIR, fi_tmp))
        os.makedirs(je.FLASHINFER_JIT_DIR, exist_ok=True)
        for name in os.listdir(prebuilt) if os.path.isdir(prebuilt) else []:
            if name != "tmp":
                os.symlink(os.path.join(prebuilt, name), os.path.join(je.FLASHINFER_JIT_DIR, name))
        if not all(s.jit_library_path.exists() for s in FIC.specs((D,))):
            raise RuntimeError("FlashInfer modules not pre-built (tools/build_flashinfer_cache.py)")
        orig = jc.JitSpec.build
        jc.JitSpec.build = lambda self, verbose, need_lock=True: None if self.jit_library_path.exists() else orig(self, verbose, need_lock)
        ws = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        q3 = runner.qkv[:, :runner.q_size].view(-1, HQ, D)
        o3 = runner.attn_out.view(-1, HQ, D)
        L = cfg.num_layers
        ours = [lambda li=li: ops.batch_decode(runner.plan, q3, runner.k_caches[li], runner.v_caches[li], runner.kv_indptr,
                                               runner.kv_indices, runner.kv_last, sc, o3) for li in range(L)]
        t_ours = _events_chained(torch, ours)
        npg = (ctx + cfg.block_size - 1) // cfg.block_size
        for tc in (True, False):
            name = (f"paged decode attention B=1 ctx={ctx} {HQ}/{HKV}x{D} vs FlashInfer fa2 (use_tensor_cores={tc}"
                    f"{', the path the reference takes for GQA>=4' if tc else ''})")
            try:
                w = flashinfer.BatchDecodeWithPagedKVCacheWrapper(ws, "NHD", use_tensor_cores=tc)
                w.plan(runner.kv_indptr[:2], runner.kv_indices[:npg], runner.kv_last[:1], HQ, HKV, D, cfg.block_size,
                       pos_encoding_mode="NONE", q_data_type=BF16, kv_data_type=BF16, sm_scale=sc)
                theirs = [lambda li=li: w.run(q3, (runner.k_caches[li], runner.v_caches[li]), out=o3) for li in range(L)]
                add(name, t_ours, _events_chained(torch, theirs),
                    "mean of 28 back-to-back launches over 28 layers' caches (235 MB > L2); FlashInfer time includes its "
                    "Python wrapper dispatch")
            except Exception as e:      # e.g. the CUDA-core decode kernel is not instantiated for GQA group 7
                out.append({"name": name, "error": str(e).strip().splitlines()[-1][:160]})
        Mp, Sp = 8192, 2048
        qkv_p = torch.randn(Mp, cfg.q_size + 2 * cfg.kv_size, device=dev, dtype=BF16)
        cu = torch.arange(0, Mp + 1, Sp, dtype=torch.int32, device=dev)
        o_p = torch.empty(Mp, HQ, D, device=dev, dtype=BF16)
        qp = qkv_p[:, :cfg.q_size].view(Mp, HQ, D)
        kp = qkv_p[:, cfg.q_size:cfg.q_size + cfg.kv_size].view(Mp, HKV, D)
        vp = qkv_p[:, cfg.q_size + cfg.kv_size:].view(Mp, HKV, D)
        wp = flashinfer.BatchPrefillWithRaggedKVCacheWrapper(ws, "NHD", backend="fa2")
        wp.plan(cu, cu, HQ, HKV, D, causal=True, pos_encoding_mode="NONE", sm_scale=sc, q_data_type=BF16, kv_data_type=BF16)
        t_o = _time_fn(torch, lambda: ops.batch_prefill(qp, kp, vp, cu, cu, sc, o_p, None, max_qo_len=Sp)) * 1e6
        t_t = _time_fn(torch, lambda: wp.run(qp, kp, vp, out=o_p)) * 1e6
        add(f"ragged causal prefill attention 4x{Sp} {HQ}/{HKV}x{D} vs FlashInfer fa2", t_o, t_t)
    except Exception as e:
        out.append({"name": "FlashInfer fa2 attention", "error": str(e)[:200]})
    finally:
        shutil.rmtree(fi_tmp, ignore_errors=True)
    # ---- linears: cuBLASLt bf16 and torch._scaled_mm fp8 at the four projection shapes, M = 8192 ----------------------
    try:
        import torch.nn.functional as F
        M = 8192
        shapes = {"qkv": (cfg.q_size + 2 * cfg.kv_size, cfg.hidden_size), "o": (cfg.hidden_size, cfg.q_size),
                  "gate_up": (2 * cfg.intermediate_size, cfg.hidden_size), "down": (cfg.hidden_size, cfg.intermediate_size)}
        for name, (N, K) in shapes.items():
            a = torch.randn(M, K, device=dev, dtype=BF16)
            wt = torch.randn(N, K, device=dev, dtype=BF16) * 0.02
            y = torch.empty(M, N, device=dev, dtype=BF16)
            t_o = _time_fn(torch, lambda: ops.gemm_bf16(a, wt, None, y)) * 1e6
            t_t = _time_fn(torch, lambda: F.linear(a, wt)) * 1e6
            add(f"bf16 linear {name} {M}x{N}x{K} vs F.linear (cuBLASLt, the reference's matmul)", t_o, t_t)
            a8, w8 = a.to(torch.float8_e4m3fn), wt.clamp(-1, 1).to(torch.float8_e4m3fn)
            one = torch.ones(1, device=dev, dtype=torch.float32)
            t_o = _time_fn(torch, lambda: ops.cutlass_scaled_mm(y, a8, w8.t(), one, one, None)) * 1e6
            t_t = _time_fn(torch, lambda: torch._scaled_mm(a8, w8.t(), scale_a=one, scale_b=one, out_dtype=BF16)) * 1e6
            add(f"fp8 scaled mm {name} {M}x{N}x{K} vs torch._scaled_mm (stand-in for cutlass_scaled_mm)", t_o, t_t)
            del a, wt, y, a8, w8
    except Exception as e:
        out.append({"name": "library GEMMs", "error": str(e)[:200]})
    return out


def scale_target_llama70b(torch, dist, dev, rank, world, exchange, steps=8, warmup=3, batch=32, ctx=8192):
    """The configuration the north-star's scaling target is defined on (BASELINE.json configs[3]): Llama-3-70B FP8 (W8A8,
    per-tensor static scales: fp8_linear_forward, linear.cpp:137-182), batch 32, ctx 8192, decode step, TP = N over the
    world group (64 q / 8 kv heads divide by 1, 2, 4, 8).  Random-init weights of the architecture, KV N(0,1).  Returns
    a dict for the extra key "scale_target" (collective: every rank calls it); an {"error": ...} dict when the box
    cannot hold the shard."""
    from xllm_b200.parallel import ProcessGroup
    from xllm_b200.qwen2 import Qwen2Config, Qwen2DecodeRunner, Qwen2Weights
    cfg = Qwen2Config.llama3_70b()
    tp = world
    out = {"workload": f"Llama-3-70B FP8 W8A8 (static per-tensor), batch={batch}, ctx={ctx}, decode step, tp{tp}", "tp": tp,
           "n_gpus": world, "steps": steps}
    try:
        torch.cuda.empty_cache()
        free, _total = torch.cuda.mem_get_info()
        per_layer = ((cfg.q_size + 2 * cfg.kv_size) * cfg.hidden_size + cfg.hidden_size * cfg.q_size +
                     3 * cfg.intermediate_size * cfg.hidden_size) // tp
        kv = cfg.num_layers * 2 * (batch * (ctx // cfg.block_size) + 1) * cfg.block_size * max(1, cfg.n_kv_heads // tp) * cfg.head_dim * 2
        need = cfg.num_layers * per_layer + kv + 2 * cfg.vocab_size * cfg.hidden_size * 2 // max(1, tp) + (6 << 30)
        out["bytes_needed_per_gpu"] = need
        ok = torch.tensor([1.0 if free > need else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() < 0.5:
            out["error"] = f"needs {need / 2**30:.0f} GiB per GPU, {free / 2**30:.0f} GiB free"
            return out
        pg = ProcessGroup() if world > 1 else None
        weights = Qwen2Weights.synthetic(cfg, dev, seed=2026, tp_rank=rank if world > 1 else 0, tp=tp)
        runner = Qwen2DecodeRunner(cfg, weights, max_batch=batch, max_ctx=ctx, device=dev, pg=pg, exchange=exchange)
        g = torch.Generator(device=dev).manual_seed(11 + rank)
        for li in range(cfg.num_layers):
            runner.k_caches[li].normal_(generator=g)
            runner.v_caches[li].normal_(generator=g)
        bs = cfg.block_size
        npg = ctx // bs
        perm = (torch.randperm(runner.num_blocks - 1, generator=torch.Generator().manual_seed(2026)) + 1).tolist()
        pages, indptr, slots = [], [0], []
        for b in range(batch):
            pb = perm[b * npg:(b + 1) * npg]
            pages += pb
            indptr.append(len(pages))
            slots.append(pb[(ctx - 1) // bs] * bs + (ctx - 1) % bs)
        runner.set_inputs_host(list(range(100, 100 + batch)), [ctx - 1] * batch, slots, indptr, pages, [(ctx - 1) % bs + 1] * batch)
        runner.step()
        runner.capture()
        for _ in range(warmup):
            runner.run_device_only()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            runner.run_device_only()
            runner.token_ids.copy_(runner.next_tokens)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0]) / steps
        step_bytes = weights.weight_bytes() + cfg.num_layers * 2 * batch * ctx * runner.nkv * cfg.head_dim * 2
        peak, _ = load_peaks()
        out.update({"tokens_per_s": batch / (ms / 1e3), "ms_per_step": ms, "step_bytes_per_gpu": step_bytes,
                    "hbm_frac_per_gpu": step_bytes / ms / 1e6 / peak, "exchange": runner.exchange_mode if world > 1 else None,
                    "timing": "CUDA events around the replays of one CUDA graph per rank, max over ranks"})
        del runner, weights
        torch.cuda.empty_cache()
    except Exception as e:                                   # the headline line must still be printed
        out["error"] = f"{type(e).__name__}: {str(e)[:160]}"
    return out


def dump_outputs(out_dir, runner):
    """what a caller of the timed decode step receives from its last replay: the logits (float32 [batch, vocab], every
    vocabulary column) and the greedy next token ids (float64, exact).  Rank 0 only: under TP its logits are the gathered
    ones; with several replicas, replica 0's."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), runner.logits.float().cpu().numpy())
    np.save(os.path.join(out_dir, "next_tokens.npy"), runner.next_tokens.cpu().numpy().astype(np.float64))


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-comparators", action="store_true")
    ap.add_argument("--ctx", type=int, default=CTX)
    ap.add_argument("--parallelism", default="tp", choices=["tp", "dp"])
    ap.add_argument("--tp", type=int, default=0, help="tensor-parallel degree (default: min(N, 4) for Qwen2-7B's 28 heads)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"])
    ap.add_argument("--no-scale-target", action="store_true", help="skip the Llama-3-70B FP8 batch-32 ctx-8192 measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step returned (logits, "
                                                          "next token ids) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import faulthandler
    import torch
    import torch.distributed as dist
    from xllm_b200 import _lib
    # watchdog: dump every thread's stack and exit if the run has not finished after `wd` seconds.  On by default for
    # multi-rank runs (a wedged collective must fail the run, not hang the box); XB_BENCH_WATCHDOG=0 disables it.
    wd = int(os.environ.get("XB_BENCH_WATCHDOG", "600" if world > 1 else "0"))
    if wd > 0:
        faulthandler.dump_traceback_later(wd, exit=True)

    def log(msg):
        if os.environ.get("XB_BENCH_VERBOSE"):
            sys.stderr.write(f"[bench rank {rank}] {msg}\n")
            sys.stderr.flush()
    from xllm_b200 import ops
    from xllm_b200.qwen2 import Qwen2Config, Qwen2DecodeRunner, Qwen2Weights
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a short timeout turns a rendezvous problem into an error (and the NCCL fallback below) instead of a hang
        dist.init_process_group("nccl", device_id=torch.device(dev), timeout=datetime.timedelta(seconds=240))
    log("process group ready")
    _lib.lib()                      # fail loudly if the CUDA library is missing: no fallback
    peak_gbs, peak_src = load_peaks()

    cfg = Qwen2Config.qwen2_7b()
    ctx = args.ctx
    tp = 1
    if world > 1 and args.parallelism == "tp":
        tp = args.tp if args.tp > 0 else (4 if world % 4 == 0 else (2 if world % 2 == 0 else 1))
        assert world % tp == 0 and cfg.n_heads % tp == 0, f"tp {tp} must divide world {world} and {cfg.n_heads} q heads"
    dp = world // tp
    pg = None
    exchange = args.exchange
    tp_parity = None
    if tp > 1:
        from xllm_b200.parallel import make_tp_group
        from xllm_b200.tp_check import tp_parity as run_tp_parity
        # dp == 1: the default group; dp > 1: one sub-group per replica (symmetric-memory rendezvous on the sub-group)
        pg = make_tp_group(rank, world, tp)
        # TP correctness first (tiny config, same exchange + CUDA graph as the timed run): TP logits vs single GPU
        tp_parity = run_tp_parity(pg, dev, exchange)
        log(f"tp parity {tp_parity}")
        ok = tp_parity["rel_l2"] <= 2e-2 and tp_parity["tokens_equal"] and tp_parity["ranks_bit_identical"]
        if not ok:
            if rank == 0:
                print(json.dumps({"error": "tp_parity failed", "tp_parity": tp_parity}), flush=True)
            sys.stdout.flush()
            os._exit(3)
    tp_rank = rank % tp
    dp_index = rank // tp
    # replicated tensors (embedding, norms) share the seed within a TP group; shards are seeded per rank
    weights = Qwen2Weights.synthetic(cfg, dev, seed=2026 + dp_index, tp_rank=tp_rank, tp=tp)
    runner = Qwen2DecodeRunner(cfg, weights, max_batch=1, max_ctx=ctx, device=dev, pg=pg, exchange=exchange)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    for li in range(cfg.num_layers):
        runner.k_caches[li].normal_(generator=g)
        runner.v_caches[li].normal_(generator=g)
    bs = cfg.block_size
    npg = (ctx + bs - 1) // bs
    pages = (torch.randperm(runner.num_blocks - 1, generator=torch.Generator().manual_seed(2026)) + 1)[:npg].tolist()
    pos = ctx - 1
    slot = pages[pos // bs] * bs + pos % bs
    tok = 1234
    runner.set_inputs_host([tok], [pos], [slot], [0, npg], pages, [(ctx - 1) % bs + 1])
    log("runner built")
    runner.step()                   # eager pass (module load, attribute setup)
    log("eager step done")
    runner.capture()
    log("graph captured")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timed region ------------------------------------------------------------------------
    for _ in range(args.warmup):
        runner.run_device_only()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        runner.run_device_only()
        runner.token_ids.copy_(runner.next_tokens)        # greedy feedback keeps the data dependency real (device op)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    log(f"timed region done: {ms:.1f} ms")
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, runner)
    # a graph replay does not pass through the library's launch counter: count the kernels in one step eagerly
    n0 = _lib.launch_count()
    runner.launch_step()
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - n0

    # ---- end-to-end region (host buffers, H2D + D2H inside) -----------------------------------------------------
    for _ in range(3):
        runner.step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = runner.step()
        runner.h_token_ids[0] = int(out[0]) % cfg.vocab_size
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    log("e2e region done")

    # ---- dominant kernel: W4A16 gate_up GEMV + SiLU*mul epilogue (the variant the graph runs) ----------------------
    L = weights.layers

    def gate_up_fn(li):
        gu = L[li]["gate_up"]
        if gu.kind == "w4a16" and gu.gate_up_interleaved and runner.fuse_gemv and tp == 1:
            # exactly the launch _launch_step_fused() makes: split-RMSNorm consumer prologue + SiLU*mul epilogue
            return lambda: ops.w4a16_decode_fused(runner.res_pp[0], gu.qweight, gu.meta, gu.group_size, gu.bias, runner.act,
                                                  norm_weight=L[li]["post_norm"], eps=cfg.rms_norm_eps,
                                                  norm_stats_in=runner.norm_stats[0], epilogue="act_mul", act_mode="silu")
        if gu.kind == "w4a16" and gu.gate_up_interleaved:
            return lambda: ops.w4a16_gate_up_act(runner.buf_a, gu.qweight, gu.meta, gu.group_size, "silu", gu.bias, runner.act,
                                                 runner.gate_up)
        return lambda: gu.forward(runner.buf_a, runner.gate_up)
    gu_fns = [gate_up_fn(li) for li in range(cfg.num_layers)]
    gu_us_avg, gu_us_med = _events_per_launch(torch, gu_fns)
    gu_us_chained = _events_chained(torch, gu_fns)
    gu = L[0]["gate_up"]
    gu_N, gu_K = gu.N, gu.K
    fused_act = gu.kind == "w4a16" and gu.gate_up_interleaved
    n_out = gu.N // 2 if fused_act else gu.N
    gu_bytes = gu.qweight.numel() * 4 + gu.meta.numel() * 4 + gu.K * 2 + n_out * 2      # this rank's shard
    # ---- the decode attention kernel the north-star names ----------------------------------------------------------
    q3 = runner.qkv[:, :runner.q_size].view(-1, runner.nh, cfg.head_dim)
    o3 = runner.attn_out.view(-1, runner.nh, cfg.head_dim)
    at_fns = [lambda li=li: ops.batch_decode(runner.plan, q3, runner.k_caches[li], runner.v_caches[li], runner.kv_indptr,
                                             runner.kv_indices, runner.kv_last, cfg.head_dim ** -0.5, o3)
              for li in range(cfg.num_layers)]
    at_us_iso, _ = _events_per_launch(torch, at_fns)
    at_us_chained = _events_chained(torch, at_fns)
    at_bytes = 2 * ctx * runner.nkv * cfg.head_dim * 2 + 2 * runner.nh * cfg.head_dim * 2 + 4 * npg

    # ---- prefill half of the metric (BASELINE.json: "... + prefill TFLOPS"): one decoder layer of the chunked-prefill
    # shape of configs[2] (4 prompts x 2048 tokens per chunk): the four W4A16 tcgen05 GEMMs + causal prefill attention ----
    prefill = None
    comparators = None
    if rank == 0 and tp == 1:
        try:
            Mp, Sp = 8192, 2048
            xin = torch.randn(Mp, cfg.hidden_size, device=dev, dtype=torch.bfloat16)
            l0 = L[0]
            bufs = {k: torch.empty(Mp, l0[k].N, device=dev, dtype=torch.bfloat16) for k in ("qkv", "o", "gate_up", "down")}
            xi = {"qkv": xin, "o": torch.randn(Mp, l0["o"].K, device=dev, dtype=torch.bfloat16), "gate_up": xin,
                  "down": torch.randn(Mp, l0["down"].K, device=dev, dtype=torch.bfloat16)}
            qkv_p = torch.randn(Mp, cfg.q_size + 2 * cfg.kv_size, device=dev, dtype=torch.bfloat16)
            cu = torch.arange(0, Mp + 1, Sp, dtype=torch.int32, device=dev)
            o_p = torch.empty(Mp, cfg.n_heads, cfg.head_dim, device=dev, dtype=torch.bfloat16)

            def gemms():
                for k in ("qkv", "o", "gate_up", "down"):
                    ops.gemm_w4a16(xi[k], l0[k].qweight, l0[k].meta, cfg.group_size, None, bufs[k])

            def attn():
                ops.batch_prefill(qkv_p[:, :cfg.q_size].view(Mp, cfg.n_heads, cfg.head_dim),
                                  qkv_p[:, cfg.q_size:cfg.q_size + cfg.kv_size].view(Mp, cfg.n_kv_heads, cfg.head_dim),
                                  qkv_p[:, cfg.q_size + cfg.kv_size:].view(Mp, cfg.n_kv_heads, cfg.head_dim), cu, cu,
                                  cfg.head_dim ** -0.5, o_p, None, max_qo_len=Sp)
            tg, ta = _time_fn(torch, gemms), _time_fn(torch, attn)
            gflop = 2.0 * Mp * sum(l0[k].N * l0[k].K for k in ("qkv", "o", "gate_up", "down"))
            aflop = 4.0 * cfg.n_heads * cfg.head_dim * Sp * Sp / 2 * (Mp // Sp)
            try:
                tf_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
            except Exception:
                tf_peak = 1400.0
            prefill = {"workload": "one Qwen2-7B decoder layer, chunk of 4 x 2048 tokens (W4A16 linears + causal attention)",
                       "linear_tflops": gflop / tg / 1e12, "linear_frac_of_bf16_sustained": gflop / tg / 1e12 / tf_peak,
                       "attention_tflops_causal": aflop / ta / 1e12, "layer_tflops": (gflop + aflop) / (tg + ta) / 1e12,
                       "prefill_tokens_per_s_extrapolated": Mp / ((tg + ta) * cfg.num_layers), "bf16_peak_tflops": tf_peak}
            del xin, bufs, xi, qkv_p, o_p, l0
        except Exception as e:      # the decode line must still be printed
            prefill = {"error": str(e)[:200]}
        if not args.no_comparators:
            try:
                comparators = gpu_comparators(torch, ops, cfg, runner, weights, dev, ctx)
            except Exception as e:
                comparators = [{"error": str(e)[:200]}]

    plan_info = (runner.plan.chunk_tokens, runner.plan.max_splits, runner.plan.cluster)
    exch_mode = runner.exchange_mode if tp > 1 else None
    h2d, d2h = runner.h2d_bytes, runner.d2h_bytes
    weights_bytes = weights.weight_bytes()

    # ---- reduce over ranks ----------------------------------------------------------------------------------------
    t = torch.tensor([ms, e2e_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    total_tokens = args.steps * dp
    value = total_tokens / (ms / 1e3)
    e2e_value = total_tokens / (e2e_ms / 1e3)
    step_bytes = weights_bytes + cfg.num_layers * at_bytes      # per rank

    def emit(scale_target, with_cpu=True):
        """rank 0: build and print THE JSON line (called once)."""
        cpu = None
        if with_cpu and not args.no_cpu_baseline:
            tps, step_s, threads, sample, spread = cpu_layer_baseline(budget_s=15.0)
            cpu = {"value": tps, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "spread": spread}
        ach = gu_bytes / gu_us_avg / 1e3
        traffic_file = "r02_w4_gemv_gateup.md"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True,
            # tensor parallelism splits ONE request's step over the GPUs of a group (strong scaling, the reference's TP);
            # N = 8 runs two TP4 groups (28 q heads do not divide by 8), each decoding its own request
            "scaling": "strong" if args.parallelism == "tp" else "weak",
            "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "ctx": ctx, "batch": 1,
                       "parallelism": (f"tp{tp}" if dp == 1 else f"tp{tp}xdp{dp}") if tp > 1 else f"dp{world}",
                       "exchange": exch_mode,
                       "l2": "inputs larger than L2: each step streams %.2f GB of weights+KV" % (step_bytes / 1e9),
                       "decode_chunk_tokens": plan_info[0], "decode_splits": plan_info[1],
                       "decode_cluster": plan_info[2], "launches_per_step": launches_per_step},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "hbm",
                         "kernel": f"linear_w4a16_small_m_kernel{' + SiLU*mul epilogue' if fused_act else ''} "
                                   f"(gate_up_proj {gu_N}x{gu_K}, 28 launches/step)",
                         "per_rank": True, "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs,
                         # ncu dram__bytes_read+write of the same kernel variant and shape (single GPU, unsharded shape)
                         "traffic": profiled_traffic(traffic_file) if tp == 1 else None,
                         "traffic_source": f"profiles/{traffic_file} (committed ncu --set full summary; cross-reference)",
                         "peak_source": peak_src, "launch_us": gu_us_avg, "launch_us_median": gu_us_med,
                         "launch_us_chained": gu_us_chained, "bytes_per_launch": gu_bytes,
                         "method": "CUDA events around each of 2 x 28 launches (one per layer's weights: 1.9 GB > L2)",
                         "step": {"bytes": step_bytes, "achieved": step_bytes / (ms / args.steps) / 1e6,
                                  "frac": step_bytes / (ms / args.steps) / 1e6 / peak_gbs},
                         "paged_decode": {"bytes_per_launch": at_bytes, "launch_us": at_us_chained,
                                          "launch_us_isolated": at_us_iso,
                                          "achieved": at_bytes / at_us_chained / 1e3,
                                          "frac": at_bytes / at_us_chained / 1e3 / peak_gbs,
                                          "frac_isolated": at_bytes / at_us_iso / 1e3 / peak_gbs,
                                          "method": "launch_us = mean over 5 x 28 back-to-back launches (one per layer's "
                                                    "KV cache, 235 MB > L2), PDL-chained as inside the decode step, one "
                                                    "event pair around the batch; launch_us_isolated = event pair "
                                                    "around every single launch"}},
            "cpu_baseline": cpu,
            "prefill": prefill,
        }
        if tp_parity is not None:
            line["tp_parity"] = tp_parity
        if comparators is not None:
            line["comparators"] = comparators
        if scale_target is not None:
            line["scale_target"] = scale_target
        print(json.dumps(line), flush=True)

    # ---- the configuration the 1 -> 8 scaling target is defined on (extra key; the headline stays Qwen2-7B) ----------
    # It builds a second model and (N > 1) a second symmetric-memory rendezvous on the world group: a guard timer makes
    # sure the headline line is printed even if that extra measurement wedges (scale_target then carries the error).
    scale_target = None
    if not args.no_scale_target and args.parallelism == "tp" and world in (1, 2, 4, 8):
        # release the Qwen2-7B runner (weights, caches, graph) before the 70B shard is built
        runner = weights = L = gu = q3 = o3 = at_fns = gu_fns = gate_up_fn = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        guard_s = float(os.environ.get("XB_SCALE_TARGET_TIMEOUT", "300"))

        def bail():
            if rank == 0:
                emit({"error": f"scale target did not finish within {guard_s:.0f} s (headline unaffected)"}, with_cpu=False)
            sys.stdout.flush()
            os._exit(0)
        guard = threading.Timer(guard_s, bail)
        guard.daemon = True
        guard.start()
        scale_target = scale_target_llama70b(torch, dist, dev, rank, world, exchange)
        guard.cancel()
        log(f"scale target {scale_target}")
    if rank == 0:
        emit(scale_target)
    if world > 1:
        # destroy_process_group() blocks here (captured NCCL / symmetric-memory graphs still hold communicator
        # references); every rank is done and rank 0 has printed, so leave without the collective teardown
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)


if __name__ == "__main__":
    main()
