#!/usr/bin/env python
"""bench.py -- ChatTS-14B decode tokens/s on B200 (BASELINE.json metric), with roofline, e2e and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl b200|reference]

One JSON line on stdout (rank 0).  A "step" is one decode step of the whole batch (one new token per
sequence) of ChatTS-14B (synthetic bf16 weights at the real shapes -- no checkpoint exists offline) after a
prefill of prompts that each carry 8 series x 256 points (8 x (46 prefix ids + <ts> + 16 patch rows + <ts/>)
+ 64 prompt ids = 576 merged positions).  `value` = B*K / device time of K steps (CUDA events, inputs
resident in HBM; the 28 GB weight stream is far larger than the 126 MB L2).  `e2e` = the same metric through
the public generate() call with HOST tensors (processor output on the CPU, H2D of ids/series, prefill, K new
tokens streamed back D2H every step).  N>1: tensor parallel over N GPUs (strong scaling, total work fixed).
At N=1 a guarded probe (two child runs of this script on 4 layers) decides whether the measured run uses the cluster-fused decode GEMMs:
only if they reproduce the default path's greedy tokens for every batch, faster (probe_decode_variant; --no-probe skips it).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SERIES, SERIES_LEN, PREFIX_IDS, PROMPT_IDS = 8, 256, 46, 64
PROMPT_POSITIONS = N_SERIES * (PREFIX_IDS + 2 + SERIES_LEN // 16) + PROMPT_IDS          # 576 merged positions per prompt
DUMP_BYTES = 64 << 20                                                                   # --dump-outputs: at most this much in all


def seq_capacity(max_new, prompt_positions=PROMPT_POSITIONS):
    """KV positions per sequence of a benchmark model: 1024, or more when --steps asks for more new tokens than that holds."""
    return max(1024, -(-(prompt_positions + max_new) // 64) * 64)


def dump_outputs(out_dir, logits, tokens):
    """--dump-outputs: what the timed decode path hands its caller after its last step -- the next-token logits of every sequence
    [B, V] and every greedy token generated so far [B, n] -- as out_dir/logits.npy (float32) and out_dir/tokens.npy (float64, exact).
    Logits larger than what DUMP_BYTES leaves keep a fixed, seeded sample of vocabulary columns (the same columns for every
    sequence), whose indices go to out_dir/logits_columns.npy.  Returns the names written."""
    os.makedirs(out_dir, exist_ok=True)
    tok = tokens.cpu().numpy().astype(np.float64)
    lg = logits.float().cpu().numpy()
    out = {"tokens": tok, "logits": lg}
    room = (DUMP_BYTES - tok.nbytes) // (4 * lg.shape[0] + 8)
    if lg.shape[1] > room:
        cols = np.sort(np.random.default_rng(0).choice(lg.shape[1], room, replace=False))
        out["logits"], out["logits_columns"] = np.ascontiguousarray(lg[:, cols]), cols.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(out)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json, cuBLAS bf16 burst)"
    return 1700.0, "fallback (B200_PROFILING.md)"


def _event_timer(fn, reps):
    """us per call of fn(i), i = 0..reps-1, between CUDA events on the current stream (after one untimed pass)."""
    fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def measure_attention(model, st, batch, ctx_len, prompt_len, hbm_peak, timer=_event_timer):
    """north_star: "attention tensor-pipe util reported as achieved fraction of roofline".  Both attention kernels timed
    ALONE on the launching stream:
      * paged flash-decode at the benchmark batch / context, one launch per LAYER's cache (48 x 84 MB at b=32 >> L2, so every
        launch streams its K/V from HBM) -> GB/s against the HBM peak (GQA intensity nh/nkv flop/B: HBM-bound);
      * tcgen05 prefill attention over batch x prompt_len positions (Q/K/V/O 0.28 GB > L2) -> causal-useful TFLOP/s
        (4 * S^2/2 * d * nh per sequence) against the measured bf16 tensor peak."""
    import math
    c, L = model.ctx, model.L
    nh, nkv, d = model.nh, model.nkv, model.d
    scale = 1.0 / math.sqrt(d)
    dev, dt = model.device, model.dtype
    out = {}
    # ---- decode: st.page_table / st.seq_lens still describe the benchmark batch (pages keep their contents after release)
    us = timer(lambda i: c.attn_decode(st.q, model.kv[i % L, 0], model.kv[i % L, 1], st.page_table, st.seq_lens, batch, nh, nkv, d,
                                       model.page_size, scale, st.attn_splits, st.attn_ws, st.ao), 2 * L)
    alg = batch * ctx_len * 2 * nkv * d * 2 + 2 * batch * nh * d * 2
    out["decode"] = {"kernel": "attn_decode_kernel (TMA paged flash-decode, mma.sync, fused split merge)", "bound": "hbm", "us_per_launch": us,
                     "algorithmic_bytes": alg, "achieved_gbs": alg / (us * 1e-6) / 1e9, "frac": alg / (us * 1e-6) / 1e9 / hbm_peak,
                     "batch": batch, "context": ctx_len, "splits": st.attn_splits}
    # ---- prefill
    T = batch * prompt_len
    g = torch.Generator(device=dev).manual_seed(7) if str(dev) != "cpu" else torch.Generator().manual_seed(7)
    q = (torch.randn(T, nh * d, device=dev, generator=g) * 0.5).to(dt)
    k = (torch.randn(T, nkv * d, device=dev, generator=g) * 0.5).to(dt)
    v = (torch.randn(T, nkv * d, device=dev, generator=g) * 0.5).to(dt)
    o = torch.empty(T, nh * d, device=dev, dtype=dt)
    cu = torch.arange(0, T + 1, prompt_len, dtype=torch.int32, device=dev)
    us = timer(lambda i: c.attn_prefill(q, k, v, cu, batch, prompt_len, nh, nkv, d, scale, o), 8)
    flops = batch * 4.0 * (prompt_len * prompt_len / 2.0) * d * nh
    peak, src = tensor_peak()
    out["prefill"] = {"kernel": "attn_prefill_tc5_kernel (tcgen05, single-pass online softmax, S/O in TMEM)" if d == 128 else "attn_prefill_kernel (HMMA)",
                      "bound": "tensor", "us_per_launch": us, "causal_flops": flops, "achieved_tflops": flops / (us * 1e-6) / 1e12,
                      "frac": flops / (us * 1e-6) / 1e12 / peak, "peak_tflops": peak, "peak_source": src, "tokens": T,
                      "tensor_pipe_active_pct_ncu": None}
    # ---- the same prefill shape through the attention kernels INSTALLED on the box (SURVEY.md 2.2 K8: "the kernel to beat"): a stated
    # comparison only -- library code, never on the product path.  Each candidate is optional (import / arch support may be missing).
    out["prefill"]["vs_installed"] = installed_attention(q, k, v, batch, prompt_len, nh, nkv, d, scale, flops, timer)
    try:       # tensor-pipe utilisation of the same kernel from the committed `ncu --set full` capture (a profiler number, never a timing)
        cap = json.load(open(os.path.join(ROOT, "profiles", "r1_ncu_summary.json")))
        out["decode"]["dram_pct_of_peak_ncu"] = float(cap["decode_attention_b32_ctx576"][0]["dram_pct_of_peak"])
        cap2 = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_attention_summary.json")))      # the single-pass kernel of round 2
        out["prefill"]["tensor_pipe_active_pct_ncu"] = float(cap2["prefill_attention_tcgen05_b32x576"][0]["tensor_pipe_active_pct"])
        out["ncu_source"] = "profiles/r1_ncu_summary.json (decode), profiles/r2_ncu_attention_summary.json (prefill)"
    except Exception:
        pass
    return out



def installed_attention(q, k, v, batch, seqlen, nh, nkv, d, scale, flops, timer):
    """Causal GQA prefill attention of the benchmark shape through the library kernels present in the image -- torch SDPA (its
    flash / cuDNN back ends) and flash_attn -- timed like our kernel (CUDA events, 8 calls after a warm-up).  Returns
    {name: {"us", "tflops"} | {"error"}}; a reference point for `attention.prefill`, never part of the product path."""
    res = {}
    T = batch * seqlen
    q4 = q.view(batch, seqlen, nh, d)
    k4 = k.view(batch, seqlen, nkv, d)
    v4 = v.view(batch, seqlen, nkv, d)

    def run(name, fn):
        try:
            fn()
            torch.cuda.synchronize()
            us = timer(lambda i: fn(), 8)
            res[name] = {"us": us, "tflops": flops / (us * 1e-6) / 1e12}
        except Exception as e:  # noqa: BLE001
            res[name] = {"error": repr(e)[:160]}

    try:
        import torch.nn.functional as F
        from torch.nn.attention import SDPBackend, sdpa_kernel
        qt, kt, vt = q4.transpose(1, 2), k4.transpose(1, 2), v4.transpose(1, 2)
        for nm, be in (("torch_sdpa_flash", SDPBackend.FLASH_ATTENTION), ("torch_sdpa_cudnn", SDPBackend.CUDNN_ATTENTION)):
            def f(be=be):
                with sdpa_kernel(be):
                    return F.scaled_dot_product_attention(qt, kt, vt, is_causal=True, scale=scale, enable_gqa=True)
            run(nm, f)
    except Exception as e:  # noqa: BLE001
        res["torch_sdpa"] = {"error": repr(e)[:160]}
    try:
        from flash_attn import flash_attn_func
        run("flash_attn_2", lambda: flash_attn_func(q4, k4, v4, causal=True, softmax_scale=scale))
    except Exception as e:  # noqa: BLE001
        res["flash_attn_2"] = {"error": repr(e)[:160]}
    return res


def make_series(i, k, length=SERIES_LEN):
    """SURVEY.md §8d synthetic series: sine + trend + noise + one level shift, seeded per (sample, series)."""
    rng = np.random.default_rng(1000 * i + k)
    t = np.arange(length)
    a = rng.uniform(0.5, 50)
    s = a * np.sin(2 * np.pi * t / rng.uniform(16, 128)) + rng.uniform(-0.05, 0.05) * t + rng.normal(0, 0.1 * a, length)
    s[int(rng.uniform(length / 4, 3 * length / 4)):] += rng.choice([-2, 2]) * a
    return s


def make_batch(cfg, batch, seed=0, n_series=N_SERIES, series_len=SERIES_LEN):
    """Host-side request batch in the reference's processor output format (input_ids, attention_mask, timeseries)."""
    from chatts_b200.processor import sp_encoding
    rng = np.random.default_rng(seed)
    ids = []
    series = []
    for b in range(batch):
        row = []
        for k in range(n_series):
            row += rng.integers(0, 150000, PREFIX_IDS).tolist() + [cfg.ts_token_start_index, cfg.ts_token_start_index + 1]
            series.append(sp_encoding(make_series(b, k, series_len))[0])
        row += rng.integers(0, 150000, PROMPT_IDS).tolist()
        ids.append(row)
    ids = torch.tensor(ids, dtype=torch.long)
    ts = torch.from_numpy(np.stack(series)).to(torch.float32)          # [B*8, 512, 1]
    return {"input_ids": ids, "attention_mask": torch.ones_like(ids), "timeseries": ts}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.stop, self.index = [], False, index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([c.strip() for c in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(r[3 + j].lower().startswith("active") for r in self.rows if len(r) > 3 + j)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def cpu_decode_baseline(batch, ctx_len, steps=3, layers_sample=2, threads=None):
    """Best of {bf16, fp32} x {all logical cores, half of them}: the most favourable setting for the reference is kept."""
    ncpu = os.cpu_count() or 1
    cands = [(torch.bfloat16, ncpu), (torch.float32, ncpu)]
    if ncpu >= 16:
        cands += [(torch.bfloat16, ncpu // 2), (torch.float32, ncpu // 2)]
    best, tried, t_start = None, [], time.time()
    for dt, th in cands:
        if best is not None and time.time() - t_start > 120:
            break
        try:
            r = _cpu_decode_baseline(batch, ctx_len, steps=steps if best is None else 2, layers_sample=layers_sample, threads=th, dtype=dt)
        except Exception as e:  # pragma: no cover
            tried.append(f"{str(dt).split('.')[-1]}/{th}t: failed {type(e).__name__}")
            continue
        tried.append(f"{str(dt).split('.')[-1]}/{th}t: {r['value']:.2f} tok/s")
        if best is None or r["value"] > best["value"]:
            best = r
    best["sample"] += "; settings tried: " + ", ".join(tried)
    return best


def _cpu_decode_baseline(batch, ctx_len, steps=3, layers_sample=2, threads=None, dtype=torch.bfloat16):
    """The reference's HF path on the host cores: stock transformers Qwen2ForCausalLM (README.md:88 loads it through
    the checkpoint's subclass) at the ChatTS-14B layer shapes, bf16, KV cache of `ctx_len` positions, batch decode.
    Bounded sample: `layers_sample` of the 48 decoder layers + final norm + lm_head are instantiated and timed; the
    per-layer time is scaled linearly to 48 layers (stated in `sample`)."""
    from transformers import Qwen2Config, Qwen2ForCausalLM
    try:
        from transformers import DynamicCache
    except ImportError:  # pragma: no cover
        from transformers.cache_utils import DynamicCache
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    full_layers = 48

    def build(nl):
        c = Qwen2Config(hidden_size=5120, intermediate_size=13824, num_hidden_layers=nl, num_attention_heads=40,
                        num_key_value_heads=8, vocab_size=152064, rms_norm_eps=1e-6, rope_theta=1e6,
                        max_position_embeddings=32768, tie_word_embeddings=False)
        with torch.device("meta"):
            m = Qwen2ForCausalLM(c)
        m = m.to_empty(device="cpu").to(dtype).eval()
        g = torch.Generator().manual_seed(1234)
        with torch.no_grad():
            for p in m.parameters():
                if p.dim() == 1:
                    p.fill_(1.0)
                else:
                    # cheap deterministic fill (randn of 2.1e9 values costs ~20 s of the budget): tile a small random block
                    blk = (torch.randn(4096, generator=g) * 0.02).to(dtype)
                    p.view(-1)[: (p.numel() // 4096) * 4096].view(-1, 4096).copy_(blk)
        # rotary buffers live outside parameters and were created on meta: rebuild them
        for mod in m.modules():
            if hasattr(mod, "inv_freq") and hasattr(mod, "compute_default_rope_parameters"):
                inv, _ = mod.compute_default_rope_parameters(c, "cpu")
                mod.inv_freq = inv
                mod.original_inv_freq = inv.clone()
        return m, c

    def time_steps(nl):
        m, c = build(nl)
        cache = DynamicCache(config=c) if "config" in DynamicCache.__init__.__code__.co_varnames else DynamicCache()
        kv = torch.randn(batch, 8, ctx_len, 128).to(dtype) * 0.1
        for l in range(nl):
            cache.update(kv.clone(), kv.clone(), l)
        ids = torch.randint(0, 150000, (batch, 1))
        ts = []
        with torch.no_grad():
            for s in range(steps + 1):
                pos = torch.full((batch, 1), ctx_len + s, dtype=torch.long)
                t0 = time.perf_counter()
                out = m(input_ids=ids, past_key_values=cache, position_ids=pos, use_cache=True)
                ids = out.logits[:, -1].float().argmax(-1, keepdim=True)
                ts.append(time.perf_counter() - t0)
        del m
        return float(np.median(ts[1:]))

    t_s = time_steps(layers_sample)
    t_0 = time_steps(0) if layers_sample > 0 else 0.0          # embed + final norm + lm_head + argmax
    per_layer = max(t_s - t_0, 0.0) / max(layers_sample, 1)
    step = t_0 + per_layer * full_layers
    return {"value": batch / step, "unit": "tokens/s", "cores": threads, "kind": "reference",
            "sample": (f"stock transformers Qwen2ForCausalLM (the reference's HF CPU path, README.md:88) {str(dtype).split('.')[-1]}, {threads} threads, ChatTS-14B layer "
                       f"shapes, batch {batch}, KV context {ctx_len}: timed {layers_sample} of 48 decoder layers + embed/norm/"
                       f"lm_head over {steps} decode steps (median), per-layer time scaled x48 "
                       f"(head {t_0 * 1e3:.0f} ms, layer {per_layer * 1e3:.0f} ms)"),
            "ms_per_step": step * 1e3}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ctx_len = N_SERIES * (PREFIX_IDS + 2 + SERIES_LEN // 16) + PROMPT_IDS
    t0 = time.time()
    vals = []
    base = None
    for _ in range(max(1, min(args.steps, 2))):
        base = cpu_decode_baseline(args.batch, ctx_len, steps=3, layers_sample=2)
        vals.append(base["value"])
        if time.time() - t0 > 150:
            break
    v = float(np.median(vals))
    base["value"] = v
    kept = "fp32" if "float32" in base.get("sample", "")[:120] else "bf16"          # the setting the search kept (stated first in `sample`)
    line = {"impl": "reference", "metric": "decode_tokens_per_s", "value": v, "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": args.batch / v * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": kept, "data": "synthetic",
            "config": workload_config(args.batch, args.gpus), "cpu_baseline": base,
            "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(batch, gpus):
    return {"workload": (f"ChatTS-14B (Qwen2.5-14B shape + 5-layer TS encoder, synthetic bf16 weights) greedy decode, batch {batch}, "
                         f"each prompt {N_SERIES} series x {SERIES_LEN} points -> 576 merged positions "
                         f"({N_SERIES}x({PREFIX_IDS} prefix ids+<ts>+16 patch rows+<ts/>)+{PROMPT_IDS} prompt ids)"),
            "batch": batch, "context": 576, "parallelism": f"tp{gpus}" if gpus > 1 else "single-gpu",
            "l2_policy": "inputs larger than L2: 28 GB of weights streamed per step vs 126 MB L2"}


# ------------------------------------------------------------------------------------------------ decode-variant probe
def _probe_run(level, args, timeout=360):
    """One guarded run of this script in a child process (its own CUDA context): 4 decoder layers of the 14B shape, the benchmark batch,
    decode timing only.  Returns the child's JSON line or a dict with 'error'."""
    import subprocess
    env = dict(os.environ, CTS_DECODE_FUSED=str(level))
    cmd = [sys.executable, os.path.abspath(__file__), "--layers", "4", "--steps", "24", "--warmup", "3", "--batch", str(args.batch),
           "--no-cpu-baseline", "--sweep-only", "--no-probe"]            # all side batches too (1 and 8 use the other token-tile instantiation)
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
        lines = [ln for ln in r.stdout.split("\n") if ln.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": f"rc={r.returncode}: {(r.stderr or r.stdout)[-300:]}"}
        d = json.loads(lines[-1])
        sha = "/".join(f"{b}:{v.get('tokens_sha1')}" for b, v in sorted(d.get("by_batch", {}).items())) or d.get("tokens_sha1")
        if "None" in str(sha):
            sha = None
        return {"ms_per_step": d["ms_per_step"], "tokens_sha1": sha, "launches_per_step": d.get("launches_per_step"),
                "ms_by_batch": {b: v.get("ms_per_step") for b, v in sorted(d.get("by_batch", {}).items())}}
    except BaseException as e:  # noqa: BLE001  (a probe must never take the benchmark down)
        return {"error": repr(e)[:300]}


def _probe_compare(level, args, timeout=420):
    """Numeric guard for a variant that is not bit-identical (tools/probe_decode_variant.py in a child process): teacher-forced next-token
    logits of the variant against the default path on a 4-layer model.  Returns its JSON line or a dict with 'error'."""
    import subprocess
    cmd = [sys.executable, os.path.join(ROOT, "tools", "probe_decode_variant.py"), "--level", str(level), "--batch", str(args.batch)]
    try:
        env = {k: v for k, v in os.environ.items() if k != "CTS_DECODE_FUSED"}
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
        lines = [ln for ln in r.stdout.split("\n") if ln.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": f"rc={r.returncode}: {(r.stderr or r.stdout)[-300:]}"}
        d = json.loads(lines[-1])
        return {"max_rel": float(d["max_rel"]), "finite": bool(d["finite"]), "steps": d.get("steps")}
    except BaseException as e:  # noqa: BLE001
        return {"error": repr(e)[:300]}


def probe_decode_variant(args):
    """The cluster-fused decode GEMMs (CTS_DECODE_FUSED=1: 7 launches per layer instead of 9, bit-identical results by construction) are
    selected for the measured run ONLY IF a guarded child run of both variants on a 4-layer model of the same shapes shows the SAME
    greedy tokens (hash over every token of the batch) and a shorter step; level 2 (5 launches per layer) only if, on top of that, its
    teacher-forced logits stay within 1e-2 of the default path's and it is faster again.  Anything else -- a fault, a timeout, different
    tokens, no gain -- leaves the previous choice in place.  The outcome is recorded in the JSON line."""
    rec = {"candidates": {}, "selected": 0}
    try:
        base = _probe_run(0, args)
        rec["candidates"]["0"] = base
        if "error" in base:
            return rec
        fused = _probe_run(1, args)
        rec["candidates"]["1"] = fused
        if "error" not in fused and fused["tokens_sha1"] and fused["tokens_sha1"] == base["tokens_sha1"] and fused["ms_per_step"] < 0.98 * base["ms_per_step"]:
            # ... and no side batch may get slower
            fb, bb = fused.get("ms_by_batch") or {}, base.get("ms_by_batch") or {}
            if all(fb.get(b) is not None and bb.get(b) is not None and fb[b] <= 1.02 * bb[b] for b in bb):
                rec["selected"] = 1
        if rec["selected"] == 1:
            # level 2 (RMSNorm folded into the next projection: 5 launches per layer) is NOT bit-identical -- the statistic is summed in
            # another order -- so its guard is numeric: teacher-forced logits within 1e-2 of the default path's at every step, then faster
            cmp = _probe_compare(2, args)
            rec["candidates"]["2_numeric"] = cmp
            if "error" not in cmp and cmp["finite"] and cmp["max_rel"] <= 1e-2:
                deep = _probe_run(2, args)
                rec["candidates"]["2"] = deep
                db = deep.get("ms_by_batch") or {}
                if ("error" not in deep and deep["ms_per_step"] < 0.98 * fused["ms_per_step"] and
                        all(db.get(b) is not None and fb.get(b) is not None and db[b] <= 1.02 * fb[b] for b in fb)):
                    rec["selected"] = 2
    except BaseException as e:  # noqa: BLE001
        rec["error"] = repr(e)[:300]
    return rec



# ------------------------------------------------------------------------------------------------ tensor-parallel parity gate
def tp_parity_gate(world, rank, layers=4, batch=8, seed=77):
    """N > 1: the tensor-parallel path against the single-GPU path on the SAME weights (a `layers`-layer model of the 14B shapes, so
    that rank 0 can hold both): next-token logits of the prefill (NCCL all-reduce path) and of one decode step (peer-memory all-reduce
    path, rows whose first token agrees), greedy agreement over 8 tokens, identical tokens on every rank.  Printed in the JSON line."""
    import torch.distributed as dist
    from chatts_b200 import ChatTSConfig
    from chatts_b200.model import ChatTSForCausalLM
    cfg = ChatTSConfig.chatts_14b()
    cfg.num_hidden_layers = layers
    kw = dict(max_batch=batch, max_seq_len=1024, page_size=64)
    tp = ChatTSForCausalLM.from_synthetic(cfg, seed=seed, tp_rank=rank, tp_size=world, **kw)
    enc = make_batch(cfg, batch, seed=3)
    S = enc["input_ids"].shape[1]
    lg_tp = tp.forward(enc["input_ids"], enc["attention_mask"], enc["timeseries"]).logits[:, 0].float()
    ids2 = tp.generate(**enc, max_new_tokens=2, ignore_eos=True)                 # prefill + ONE decode step: its logits are still in the state
    shard = tp._steps[batch].logits[:batch].float().contiguous()
    parts = [torch.empty_like(shard) for _ in range(world)]
    dist.all_gather(parts, shard)
    dec_tp = torch.cat(parts, dim=-1)
    ids_tp = tp.generate(**enc, max_new_tokens=8, ignore_eos=True)
    t = ids_tp.cuda()
    lst = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(lst, t)
    same = all(torch.equal(lst[0], x) for x in lst)
    out = None
    if rank == 0:
        ref = ChatTSForCausalLM.from_synthetic(cfg, seed=seed, **kw)
        lg = ref.forward(enc["input_ids"], enc["attention_mask"], enc["timeseries"]).logits[:, 0].float()
        r2 = ref.generate(**enc, max_new_tokens=2, ignore_eos=True)
        dec = ref._steps[batch].logits[:batch].float()
        ids = ref.generate(**enc, max_new_tokens=8, ignore_eos=True)
        rows = (r2[:, S] == ids2[:, S]).nonzero().reshape(-1).to(dec.device)
        e_pre = float((lg_tp - lg).abs().max() / lg.abs().max())
        e_dec = float((dec_tp[rows] - dec[rows]).abs().max() / dec[rows].abs().max()) if rows.numel() else None
        agree = [int(next((i for i in range(8) if ids[b, S + i] != ids_tp[b, S + i]), 8)) for b in range(batch)]
        out = {"layers": layers, "batch": batch, "prefill_logits_max_rel": e_pre, "decode_logits_max_rel": e_dec, "decode_rows_compared": int(rows.numel()),
               "greedy_agreement_of_8": agree, "identical_tokens_on_all_ranks": bool(same),
               "pass": bool(same and e_pre < 2e-2 and (e_dec is None or e_dec < 2e-2))}
        del ref
    del tp
    torch.cuda.empty_cache()
    dist.barrier()
    return out

# ------------------------------------------------------------------------------------------------ B200 arm
def measure_config4(cfg, rank, world, steps, warmup, sync_all, batch=8, n_series=30, series_len=512):
    """BASELINE.json configs[3]: batch-8 decode with 30 series x 512 points per prompt (30 x (46 prefix ids + <ts> + 32 patch rows + <ts/>)
    + 64 prompt ids = 2 464 merged positions), tensor-parallel over however many GPUs the run has (the config names 8).  A second model
    instance of the same synthetic weights with a 4 096-position cache: the headline model's buffers stay as measured.  Device-timed graph
    replays as the headline, plus the same public generate() call with pinned host tensors."""
    import torch.distributed as dist
    from chatts_b200.model import ChatTSForCausalLM
    model = ChatTSForCausalLM.from_synthetic(cfg, seed=1234, tp_rank=rank, tp_size=world, max_batch=batch, max_seq_len=4096, page_size=64)
    enc = make_batch(cfg, batch, seed=4, n_series=n_series, series_len=series_len)
    max_new = steps + warmup + 8
    ids_cpu, am_cpu, counts, lay = model._prepare_inputs(enc["input_ids"], enc["attention_mask"], enc["timeseries"])
    pts, held = model._alloc_pages(lay.lens, max_new)
    try:
        sync_all()
        t0 = time.perf_counter()
        logits = model._prefill(lay, counts, enc["timeseries"], pts)
        torch.cuda.synchronize()
        prefill_s = time.perf_counter() - t0
        st = model._decode_state(batch, max_new)
        lens32 = torch.from_numpy(lay.lens.astype(np.int32))
        st.page_table.copy_(torch.from_numpy(pts)); st.positions.copy_(lens32 - 1); st.seq_lens.copy_(lens32); st.step_ptr.zero_()
        model.ctx.greedy_advance(logits, batch, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map, st.page_table, model.page_size)
        for _ in range(max(warmup, 3)):
            model._decode_step(st)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            model._decode_step(st)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        n_tok = int(st.step_ptr[0].item())
        import hashlib
        toks = st.out_tokens[:, :n_tok].to(torch.int32).cpu().numpy()
        tok_sha = hashlib.sha1(toks.tobytes()).hexdigest()[:16]
        same = True
        if world > 1:                                   # every rank must have picked the same tokens
            tt = torch.from_numpy(toks.astype(np.int64)).cuda()
            ref = tt.clone()
            dist.broadcast(ref, src=0)
            flag = torch.tensor([int(torch.equal(tt, ref))], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            same = bool(int(flag))
    finally:
        model.pool.release(held)
    encp = {k: v.pin_memory() for k, v in enc.items()}
    model.generate(**encp, max_new_tokens=4, ignore_eos=True, sync_every=1)
    sync_all()
    t0 = time.perf_counter()
    model.generate(**encp, max_new_tokens=steps, ignore_eos=True, sync_every=1)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt)
    positions = int(lay.lens.max())
    out = {"workload": f"BASELINE.json configs[3]: batch {batch} decode, {n_series} series x {series_len} points per prompt -> {positions} merged positions, tp{world}",
           "batch": batch, "context": positions, "n_gpus": world, "steps": steps, "ms_per_step": ms / steps, "tokens_per_s": batch * steps / (ms / 1e3),
           "prefill_s": prefill_s, "prefill_positions": int(lay.lens.sum()), "tokens_sha1": tok_sha, "identical_tokens_on_all_ranks": same,
           "e2e": {"value": batch * steps / dt, "unit": "tokens/s", "seconds": dt,
                   "definition": f"model.generate(**pinned_host_tensors, max_new_tokens={steps}, sync_every=1): H2D, TS encode of {batch * n_series} series, prefill, {steps} decode steps with per-step D2H"}}
    del model
    torch.cuda.empty_cache()
    return out


def measure_w4(cfg, steps, warmup, hbm_peak, batches=(1, 8, 32)):
    """GPTQ-Int4 side block (README.md:52,262-263: ChatTS-14B-GPTQ-Int4), one GPU: a third model instance whose seven projections per
    layer are 4-bit (synthetic codes / scales / zero points at the real shapes, group size 128; embeddings, norms, lm_head and the TS
    encoder stay bf16) decodes the benchmark prompts through the packed weights (cts_gemm_w4_mma) and through its own dequantised bf16
    copy: ms per step of both from CUDA events over graph replays, greedy agreement between the two."""
    from chatts_b200.model import ChatTSForCausalLM
    max_new = steps + warmup + 8
    model = ChatTSForCausalLM.from_synthetic(cfg, seed=1234, max_batch=max(batches), max_seq_len=seq_capacity(max_new), page_size=64)
    model.quantize_w4_synthetic(group_size=128)
    w4 = model.w4

    def run(batch):
        enc = make_batch(cfg, batch)
        ids_cpu, am_cpu, counts, lay = model._prepare_inputs(enc["input_ids"], enc["attention_mask"], enc["timeseries"])
        pts, held = model._alloc_pages(lay.lens, max_new)
        try:
            logits = model._prefill(lay, counts, enc["timeseries"], pts)
            st = model._decode_state(batch, max_new)
            lens32 = torch.from_numpy(lay.lens.astype(np.int32))
            st.page_table.copy_(torch.from_numpy(pts)); st.positions.copy_(lens32 - 1); st.seq_lens.copy_(lens32); st.step_ptr.zero_()
            model.ctx.greedy_advance(logits, batch, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map, st.page_table, model.page_size)
            for _ in range(max(warmup, 3)):
                model._decode_step(st)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                model._decode_step(st)
            e1.record()
            torch.cuda.synchronize()
            toks = st.out_tokens[:, : int(st.step_ptr[0])].cpu().numpy().copy()
            return e0.elapsed_time(e1) / steps, toks
        finally:
            model.pool.release(held)

    L = cfg.num_hidden_layers
    per_layer = (cfg.hidden_size * (cfg.num_attention_heads + 2 * cfg.num_key_value_heads) * cfg.head_dim + cfg.hidden_size * cfg.num_attention_heads * cfg.head_dim +
                 3 * cfg.hidden_size * cfg.intermediate_size)
    out = {"workload": "ChatTS-14B with 4-bit projections (GPTQ layout, group 128, synthetic codes), the benchmark prompts, greedy decode; W4A16 through "
                       "cts_gemm_w4_mma against the same model through its dequantised bf16 copy", "kernel": w4["kernel"], "steps": steps, "by_batch": {}}
    for b in batches:
        model.w4, model._steps = w4, {}
        ms4, t4 = run(b)
        model.w4, model._steps = None, {}
        ms16, t16 = run(b)
        n = min(t4.shape[1], t16.shape[1])
        agree = [int(next((i for i in range(n) if t4[r, i] != t16[r, i]), n)) for r in range(b)]
        w4_bytes = L * per_layer * (0.5 + 4.0 / 128) + 2 * cfg.hidden_size * cfg.vocab_size
        kv = b * 600 * L * 2 * cfg.num_key_value_heads * cfg.head_dim * 2
        out["by_batch"][str(b)] = {"w4_ms_per_step": ms4, "bf16_ms_per_step": ms16, "speedup": ms16 / ms4, "w4_tokens_per_s": b / (ms4 / 1e3),
                                   "w4_whole_step_hbm_frac": (w4_bytes + kv) / (ms4 / 1e3) / 1e9 / hbm_peak, f"min_greedy_agreement_of_{n}": int(min(agree))}
    del model
    torch.cuda.empty_cache()
    return out


def run_b200(args):
    import torch.distributed as dist
    from chatts_b200 import ChatTSConfig, _cabi
    from chatts_b200.model import ChatTSForCausalLM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    probe_record = None
    if world == 1 and args.probe and not args.sweep_only and not args.no_probe and not args.layers and "CTS_DECODE_FUSED" not in os.environ:
        probe_record = probe_decode_variant(args)
        if probe_record.get("selected"):
            os.environ["CTS_DECODE_FUSED"] = str(probe_record["selected"])          # read by the model constructor below
    tp_gate = None
    if world > 1 and not args.sweep_only and not args.layers:
        try:
            tp_gate = tp_parity_gate(world, rank)
        except Exception as e:  # pragma: no cover  (reported, never fatal for the measurement)
            tp_gate = {"error": repr(e)[:300], "pass": False}
    cfg = ChatTSConfig.chatts_14b()
    if args.layers:
        cfg.num_hidden_layers = args.layers
    hbm_peak, peak_src = peaks()
    max_new = args.steps + args.warmup + 8
    model = ChatTSForCausalLM.from_synthetic(cfg, seed=1234, tp_rank=rank, tp_size=world, max_batch=max(args.batch, 1),
                                             max_seq_len=seq_capacity(max_new), page_size=64, use_cuda_graph=not args.no_graph)
    ctx = model.ctx

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def measure_decode(batch):
        """Prefill the batch, then W untimed + K timed decode steps on the device."""
        enc = make_batch(cfg, batch)
        ids_cpu, am_cpu, counts, lay = model._prepare_inputs(enc["input_ids"], enc["attention_mask"], enc["timeseries"])
        pts, held = model._alloc_pages(lay.lens, max_new)
        try:
            logits = model._prefill(lay, counts, enc["timeseries"], pts)
            st = model._decode_state(batch, max_new)
            lens32 = torch.from_numpy(lay.lens.astype(np.int32))
            st.page_table.copy_(torch.from_numpy(pts))
            st.positions.copy_(lens32 - 1)
            st.seq_lens.copy_(lens32)
            st.step_ptr.zero_()
            ctx.greedy_advance(logits, batch, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map,
                               st.page_table, model.page_size)
            for _ in range(max(args.warmup, 3)):        # untimed warm-up steps; the first one also captures the CUDA graph
                model._decode_step(st)
            # kernels per step, counted by running the same step body eagerly once (one more untimed step)
            l0 = ctx.launches
            model._decode_body(st, True)
            per_step_launches = ctx.launches - l0
            sync_all()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                model._decode_step(st)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t)
            n_tok = int(st.step_ptr[0].item())
            ctx_end = int(lay.lens.max()) + n_tok
            import hashlib
            tok_sha = hashlib.sha1(st.out_tokens[:, :n_tok].to(torch.int32).cpu().numpy().tobytes()).hexdigest()[:16]
            if args.dump_outputs and batch == args.batch:
                logits = model._gather_vocab(st.logits[:batch])         # every rank takes part in the gather of the vocab shards
                if rank == 0:
                    dumped.extend(dump_outputs(args.dump_outputs, logits, st.out_tokens[:batch, :n_tok]))
        finally:
            model.pool.release(held)
        return ms, per_step_launches, ctx_end, tok_sha

    results, dumped = {}, []
    with ClockSampler(local) as clk:
        batches = [args.batch] if args.only_batch else sorted(set(b for b in (1, 8, args.batch) if b <= args.batch))
        for b in batches:
            ms, launches, ctx_end, tok_sha = measure_decode(b)
            results[b] = dict(ms_total=ms, ms_per_step=ms / args.steps, tokens_per_s=b * args.steps / (ms / 1e3), launches=launches, tokens_sha1=tok_sha,
                              ctx_end=ctx_end)
    clocks = clk.summary()
    main = results[args.batch]

    # ---- whole-step HBM roofline: streamed weights + KV read per step (SURVEY.md §8d)
    L = cfg.num_hidden_layers
    per_layer = (cfg.hidden_size * (cfg.num_attention_heads + 2 * cfg.num_key_value_heads) * cfg.head_dim + cfg.hidden_size * cfg.num_attention_heads * cfg.head_dim +
                 3 * cfg.hidden_size * cfg.intermediate_size)
    w_bytes = 2 * (L * per_layer + cfg.hidden_size * cfg.vocab_size) / world
    kv_tok = L * 2 * cfg.num_key_value_heads * cfg.head_dim * 2 / world
    ctx_mid = main["ctx_end"] - args.steps / 2
    step_bytes = w_bytes + args.batch * ctx_mid * kv_tok
    step_gbs = step_bytes / (main["ms_per_step"] / 1e3) / 1e9

    # ---- dominant kernel alone: gate_up tcgen05 GEMM (2*I*H weights), one launch per layer weight so every launch
    # streams a different 283 MB from HBM (>> L2), timed with CUDA events on the launching stream
    roof = None
    if world == 1:
        st = model._decode_state(args.batch, max_new)
        B = args.batch
        I = model.I
        sp = st.splits["gu"]
        n_rep = max(1, args.steps // 4)
        for _ in range(2):
            for l in range(L):
                ctx.gemm(st.xn, model.wgu[l], st.ws, epilogue=_cabi.EPI_PARTIAL_F32, split_k=sp, t=B)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_rep):
            for l in range(L):
                ctx.gemm(st.xn, model.wgu[l], st.ws, epilogue=_cabi.EPI_PARTIAL_F32, split_k=sp, t=B)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (n_rep * L)
        alg = 2 * I * cfg.hidden_size * 2 + B * cfg.hidden_size * 2 + B * I * 2
        ach = alg / (us * 1e-6) / 1e9
        traffic = None
        try:       # dram__bytes_read+write per launch of this kernel from the committed ncu --set full capture (b=32)
            if B == 32:
                traffic = json.load(open(os.path.join(ROOT, "profiles", "r1_ncu_summary.json")))["gate_up_decode_traffic_bytes_per_launch"]
        except Exception:
            traffic = None
        roof = {"bound": "hbm", "kernel": "gemm_tn_kernel (gate_up projection, tcgen05/TMA, swap-AB, split-K 2)", "achieved": ach, "peak": hbm_peak,
                "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic, "us_per_launch": us, "algorithmic_bytes": alg,
                "peak_source": peak_src, "split_k": sp,
                "whole_step": {"bytes": step_bytes, "achieved_gbs": step_gbs, "frac": step_gbs / hbm_peak}}
        if getattr(model, "use_fused_decode", 0):
            # the measured step ran the cluster-fused variant of this projection (same TMA -> tcgen05 mainloop per K split, reduction and
            # SwiGLU in the epilogue): time THAT kernel too, same weights, same algorithmic bytes
            try:
                fs = min(sp, 8)
                for l in range(L):
                    ctx.gemm_decode_fused(st.xn, model.wgu[l], _cabi.FUSED_SWIGLU, fs, B, act=st.act)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(n_rep):
                    for l in range(L):
                        ctx.gemm_decode_fused(st.xn, model.wgu[l], _cabi.FUSED_SWIGLU, fs, B, act=st.act)
                e1.record()
                torch.cuda.synchronize()
                fus = e0.elapsed_time(e1) * 1e3 / (n_rep * L)
                roof["fused_variant"] = {"kernel": "gemm_decode_fused_kernel (gate_up + cluster split-K reduction + SwiGLU)", "us_per_launch": fus,
                                         "achieved": alg / (fus * 1e-6) / 1e9, "frac": alg / (fus * 1e-6) / 1e9 / hbm_peak, "split_k": fs}
            except Exception as e:  # pragma: no cover
                roof["fused_variant"] = {"error": repr(e)[:200]}

    # ---- TS encoder alone (north_star: reported against the HBM roofline): N = 8*B series x 256 points -> 128*B patch rows,
    # L2 flushed (256 MB write) before every timed call, CUDA events around the encode (patchify + 5 tcgen05 GEMM layers)
    ts_roof = None
    if world == 1:
        def ts_case(nb):
            enc_b = make_batch(cfg, nb, seed=2)
            x_ts = enc_b["timeseries"].to("cuda", torch.bfloat16)
            flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
            tse = model.ts_encoder
            counts = tse.patch_counts(x_ts)
            host = torch.stack([counts[1], counts[2]]).cpu()
            hc = (host[0], host[1])
            l0 = ctx.launches
            feats, pc = tse.encode(x_ts, counts=counts, host_counts=hc)             # warm (kernel attributes, allocator)
            n_launch = ctx.launches - l0
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()                                               # launch-overhead-free replay of the encoder's kernels
            with torch.cuda.graph(g):
                feats, pc = tse.encode(x_ts, counts=counts, host_counts=hc)
            reps, tot_ms, rows = 8, 0.0, int(feats.shape[0])
            for it in range(reps + 2):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g.replay()
                e1.record()
                torch.cuda.synchronize()
                if it >= 2:
                    tot_ms += e0.elapsed_time(e1)
            us = tot_ms * 1e3 / reps
            H, in0, nl = tse.hidden_size, tse.input_size, tse.num_layers
            w_bytes = 2 * (in0 * H + (nl - 1) * H * H + nl * H)
            alg = w_bytes + x_ts.numel() * 2 + rows * in0 * 2 * 2 + rows * H * 2 * (2 * nl - 1)
            flops = 2.0 * rows * (in0 * H + (nl - 1) * H * H)
            ach = alg / (us * 1e-6) / 1e9
            del g, flush
            return {"series": int(x_ts.shape[0]), "points": SERIES_LEN, "patch_rows": rows, "us": us, "algorithmic_bytes": alg,
                    "achieved_gbs": ach, "hbm_frac": ach / hbm_peak, "tflops": flops / (us * 1e-6) / 1e12,
                    "bound": "hbm (weight stream)" if rows <= 280 else "tensor", "launches": n_launch,
                    "timed": "CUDA-graph replay of patchify + MLP, L2 flushed before each replay"}

        # the metric prompt (b = 1: 8 series -> 128 patch rows, HBM-bound on the 212 MB weight stream) AND the benchmark batch
        ts_roof = dict(ts_case(args.batch))
        ts_roof["cases"] = {"b1": ts_case(1), f"b{args.batch}": {k: v for k, v in ts_roof.items()}}

    # ---- attention kernels alone (north_star: attention reported as achieved fraction of its roofline)
    attn_roof = None
    if world == 1:
        try:
            attn_roof = measure_attention(model, model._decode_state(args.batch, max_new), args.batch, int(main["ctx_end"]), 576, hbm_peak)
        except Exception as e:  # pragma: no cover  (a side measurement must never cost the headline line)
            attn_roof = {"error": repr(e)}

    # ---- e2e through the public API with host tensors
    e2e = None
    if not args.sweep_only:
        # every rank runs the same public call on the same host tensors (TP ranks are SPMD); the wall time is the max over ranks
        enc = make_batch(cfg, args.batch, seed=1)
        enc = {k: v.pin_memory() for k, v in enc.items()}
        new = args.steps
        model.generate(**enc, max_new_tokens=4, ignore_eos=True, sync_every=1)          # warm
        sync_all()
        t0 = time.perf_counter()
        out = model.generate(**enc, max_new_tokens=new, ignore_eos=True, sync_every=1)  # D2H of the new ids every step
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt)
        h2d = (enc["timeseries"].numel() * 2 + 4 * 576 * args.batch * 4 + args.batch * N_SERIES * 16 * 4)
        d2h = args.batch * new * 4 + args.batch * N_SERIES * 8
        e2e = {"value": args.batch * new / dt, "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "definition": f"one step = model.generate(**host_tensors, max_new_tokens={new}) incl. H2D, TS encode, prefill of "
                             f"{args.batch}x576 positions and {new} decode steps with per-step D2H of the new ids; value = B*new/wall",
               "seconds": dt, "out_shape": list(out.shape)}

    # ---- BASELINE.json configs[3] (batch-8 decode, 30 series x 512 points) on this run's GPUs: a side block, never fatal for the headline
    config4 = None
    if not args.sweep_only and not args.layers and not args.no_config4:
        try:
            config4 = measure_config4(cfg, rank, world, args.steps, args.warmup, sync_all)
        except Exception as e:  # pragma: no cover
            config4 = {"error": repr(e)[:300]}              # shape / capacity errors are the same on every rank: all of them land here

    # ---- GPTQ-Int4 side block (one GPU: W4A16 decode weights are single-GPU)
    w4_block = None
    if world == 1 and not args.sweep_only and not args.layers and not args.no_w4:
        try:
            w4_block = measure_w4(cfg, args.steps, args.warmup, hbm_peak, batches=sorted(set(b for b in (1, 8, args.batch) if b <= args.batch)))
        except Exception as e:  # pragma: no cover
            w4_block = {"error": repr(e)[:300]}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu = cpu_decode_baseline(args.batch, 576, steps=3, layers_sample=2)
            except Exception as e:  # pragma: no cover
                cpu = {"value": None, "unit": "tokens/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e!r}"}
        line = {"metric": "decode_tokens_per_s", "value": main["tokens_per_s"], "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": workload_config(args.batch, world),
                "by_batch": {str(b): {"tokens_per_s": r["tokens_per_s"], "ms_per_step": r["ms_per_step"], "tokens_sha1": r.get("tokens_sha1")} for b, r in results.items()},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(main["launches"] * args.steps), "launches_per_step": main["launches"],
                "roofline": roof, "ts_encoder": ts_roof, "attention": attn_roof, "cpu_baseline": cpu, "arch": ctx.arch, "lib": os.path.relpath(_cabi.LIB_PATH, ROOT)}
        # which opt-in variants of the decode path this line was measured with (all off = the validated default path)
        line["config4"] = config4
        line["w4a16"] = w4_block
        line["tokens_sha1"] = main.get("tokens_sha1")          # hash of every greedy token the measured batch produced (probe: equality across variants)
        if probe_record is not None:
            line["config"]["decode_variant_probe"] = probe_record
        if args.dump_outputs:
            line["dumped_outputs"] = {"dir": args.dump_outputs, "names": dumped, "batch": args.batch}
        if world > 1:
            line["tp_parity"] = tp_gate
            # per rank and step: 2 row-parallel tails per layer, each a two-shot exchange with the flags inside the data (LL):
            # reduce-scatter of fp32 pairs (8 B on the wire per element incl. epochs) to the owners + all-gather of the rounded h
            # (4 B per element incl. epochs), (world-1)/world of it leaving the GPU
            line["nvlink_bytes_per_step_per_rank"] = int(2 * L * args.batch * cfg.hidden_size * 12 * (world - 1) / world)
        line["config"]["variants"] = {k: int(getattr(model, a, 0) or 0) for k, a in (("decode_fused", "use_fused_decode"), ("peer_ll", "use_peer_ll"),
                                                                                   ("native_step", "use_native_step"), ("decode_chain", "use_chain"))}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--layers", type=int, default=0, help="debug: fewer decoder layers (makes the number INVALID as a benchmark)")
    ap.add_argument("--only-batch", action="store_true", help="skip the b=1/8 side measurements")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run decode steps eagerly (for ncu launch lists)")
    ap.add_argument("--sweep-only", action="store_true", help="decode timing only (skip e2e)")
    ap.add_argument("--no-w4", action="store_true", help="skip the GPTQ-Int4 side block (third model instance with 4-bit projections)")
    ap.add_argument("--no-config4", action="store_true", help="skip the BASELINE configs[3] side block (second model instance, 30 x 512-point prompts)")
    ap.add_argument("--no-probe", action="store_true", help="(default) the default decode path is measured as is")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the measured batch's last-step logits and its greedy tokens as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB; seeded inputs, so two builds can be compared output for output)")
    ap.add_argument("--probe", action="store_true", help="guarded child-process probe of the cluster-fused decode variants (round 1; measured slower at b = 32 on a B200, "
                                                        "profiles/r2_decode_variants_ab.txt, so no longer on by default)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
