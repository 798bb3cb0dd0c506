#!/usr/bin/env python
"""The W4A16 prefill GEMM (cts_gemm_w4_prefill) and the 4-bit-only model mode at ChatTS-14B shapes, synthetic group-128 codes.

  projections: per projection and t in {64, 128, 576, 2464, 18432}, the new kernel next to cts_gemm on the dequantised weight, each with
               the epilogue and split factor the model uses at that t (CUDA events; the weight copies rotate over > 126 MB so the
               weight-bound small-t launches read HBM), achieved FLOP/s and weight bytes/s; outputs compared bit for bit
  model:       ChatTSForCausalLM with w4_only=True against the default GPTQ mode (dense copy + 4-bit decode copy), one model at a time:
               allocated HBM after construction, prefill seconds of the benchmark prompts (32 x 576 positions) and of BASELINE.json
               configs[3]'s 8 prompts (30 series x 512 points = 2 464 positions each), decode ms/step at b = 1, 8, 32, 64, 128, and the
               greedy tokens of every decode run (must be identical between the modes)

    python tools/bench_w4_prefill.py [--out profiles/<name>.json] [--skip-model] [--steps 20]

Writes one JSON file (default profiles/w4_prefill_bench.json) with the card name and power limit read in the same run."""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from chatts_b200 import _cabi  # noqa: E402
from chatts_b200._cabi import EPI_NONE, EPI_PARTIAL_F32, EPI_RESIDUAL, EPI_SWIGLU_IL  # noqa: E402
from chatts_b200.weights import dequantize_w4, repack_w4_mma  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:  # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(), error=str(e))


def _timed(fn, reps):
    for _ in range(3):
        fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def projections(ts, gs=128):
    c = _cabi.get_context()
    dev, dt = "cuda", torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(1)
    H, I = 5120, 13824
    shapes = {"qkv": (7168, H), "o": (H, H), "gate_up": (2 * I, H), "down": (H, I)}
    res = {}
    for name, (n, k) in shapes.items():
        w4_bytes = n * k // 2 + n * (k // gs) * 4
        dense_bytes = n * k * 2
        n4, nd = max(2, -(-300_000_000 // w4_bytes)), max(2, -(-300_000_000 // dense_bytes))
        sc = ((torch.rand(n, k // gs, generator=g, device=dev) + 0.5) * 0.01).to(dt)
        zp = torch.randint(1, 17, (n, k // gs), generator=g, device=dev, dtype=torch.uint8)
        qws = [torch.randint(0, 256, (n, k // 2), generator=g, device=dev, dtype=torch.uint8) for _ in range(max(n4, nd))]
        frag = [repack_w4_mma(q, sc, zp, gs) for q in qws[:n4]]
        dense = [dequantize_w4(q, sc, zp, gs) for q in qws[:nd]]
        bias = (torch.randn(n, generator=g, device=dev) * 0.1).to(dt) if name == "qkv" else None
        rows = {}
        for t in ts:
            x = (torch.randn(t, k, generator=g, device=dev) * 0.5).to(dt)
            if name == "gate_up":
                split = c.suggest_split(n // 2, k, t, True)
                epi = EPI_SWIGLU_IL if t > 128 else EPI_PARTIAL_F32
            else:
                split = c.suggest_split(n, k, t)
                epi = EPI_PARTIAL_F32 if split > 1 else (EPI_NONE if name == "qkv" else EPI_RESIDUAL)
            if epi == EPI_PARTIAL_F32:
                out_a = torch.empty(split, t, n, device=dev)
            else:
                out_a = torch.empty(t, n // 2 if epi == EPI_SWIGLU_IL else n, device=dev, dtype=dt)
            out_b = torch.empty_like(out_a)
            resid = (torch.randn(t, n, generator=g, device=dev)).to(dt) if epi == EPI_RESIDUAL else None
            kw = dict(bias=bias if epi in (EPI_NONE, EPI_RESIDUAL) else None, residual=resid, epilogue=epi, split_k=split, t=t)
            reps = max(5, min(200, int(2e12 // (2 * t * n * k) + 5)))
            t_w4 = _timed(lambda i: c.gemm_w4_prefill(x, frag[i % n4][0], frag[i % n4][1], n, gs, out_a, **kw), reps)
            t_d = _timed(lambda i: c.gemm(x, dense[i % nd], out_b, **kw), reps)
            c.gemm_w4_prefill(x, frag[0][0], frag[0][1], n, gs, out_a, **kw)
            c.gemm(x, dense[0], out_b, **kw)
            torch.cuda.synchronize()
            flop = 2.0 * t * n * k
            rows[str(t)] = dict(epilogue={0: "none", 3: "partial_f32", 4: "residual", 6: "swiglu_il"}[epi], split=split, reps=reps,
                                w4_us=t_w4 * 1e6, dense_us=t_d * 1e6, w4_over_dense=t_w4 / t_d,
                                w4_tflops=flop / t_w4 / 1e12, dense_tflops=flop / t_d / 1e12,
                                w4_weight_gbps=w4_bytes / t_w4 / 1e9, dense_weight_gbps=dense_bytes / t_d / 1e9,
                                bit_identical=bool(torch.equal(out_a, out_b)))
            print(name, t, rows[str(t)], flush=True)
            del x, out_a, out_b, resid
        res[name] = dict(n=n, k=k, group_size=gs, w4_weight_bytes=w4_bytes, dense_weight_bytes=dense_bytes, by_t=rows)
        del qws, frag, dense
        gc.collect()
        torch.cuda.empty_cache()
    return res


def _prefill_s(model, enc, reps=3):
    model(**enc)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        model(**enc)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def _decode(model, cfg, b, steps, warmup=3):
    enc = bench.make_batch(cfg, b, seed=11 + b)
    max_new = steps + warmup + 2
    ids_cpu, am_cpu, counts, lay = model._prepare_inputs(enc["input_ids"], enc["attention_mask"], enc["timeseries"])
    pts, held = model._alloc_pages(lay.lens, max_new)
    try:
        logits = model._prefill(lay, counts, enc["timeseries"], pts)
        st = model._decode_state(b, max_new)
        lens32 = torch.from_numpy(lay.lens.astype(np.int32))
        st.page_table.copy_(torch.from_numpy(pts)); st.positions.copy_(lens32 - 1); st.seq_lens.copy_(lens32); st.step_ptr.zero_()
        model.ctx.greedy_advance(logits, b, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map, st.page_table,
                                 model.page_size)
        for _ in range(warmup):
            model._decode_step(st)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            model._decode_step(st)
        e1.record()
        torch.cuda.synchronize()
        n_tok = int(st.step_ptr[0].item())
        return e0.elapsed_time(e1) / steps, st.out_tokens[:b, :n_tok].cpu().clone()
    finally:
        model.pool.release(held)
        model._steps.pop(b, None)


def whole_model(steps, batches=(1, 8, 32, 64, 128)):
    from chatts_b200 import ChatTSConfig
    from chatts_b200.model import ChatTSForCausalLM
    cfg = ChatTSConfig.chatts_14b()
    out, toks = {}, {}
    for mode in ("default_gptq", "w4_only"):
        gc.collect()
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        t0 = time.perf_counter()
        m = ChatTSForCausalLM.from_synthetic(cfg, seed=1234, max_batch=128, max_seq_len=2560, page_size=64)
        m.quantize_w4_synthetic(group_size=128, w4_only=(mode == "w4_only"))
        gc.collect()
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        alloc = torch.cuda.memory_allocated() - base
        tensors = [m.embed, m.lm_head, m.final_norm] + m.ln1 + m.ln2 + [t for t in m.bqkv + m.qn + m.kn if t is not None]
        tensors += [t for lst in (m.wqkv, m.wo, m.wgu, m.wd) for t in lst if t is not None]
        tensors += [t for kind in ("qkv", "o", "gu", "d") for e in m.w4[kind] for t in e if isinstance(t, torch.Tensor)]
        weights = sum(t.numel() * t.element_size() for t in tensors)
        kv = m.kv.numel() * m.kv.element_size()
        r = dict(allocated_after_construction_bytes=alloc, weight_bytes=weight_bytes_str(weights), weight_bytes_exact=weights,
                 kv_cache_bytes=kv, build_s=build_s)
        enc32 = bench.make_batch(cfg, 32, seed=0)
        r["prefill_s_32x576"] = _prefill_s(m, enc32)
        enc8 = bench.make_batch(cfg, 8, seed=4, n_series=30, series_len=512)
        r["prefill_s_config4_8x2464"] = _prefill_s(m, enc8)
        r["decode_ms_per_step"] = {}
        for b in batches:
            ms, tk = _decode(m, cfg, b, steps)
            r["decode_ms_per_step"][str(b)] = ms
            toks.setdefault(b, []).append(tk)
        print(mode, r, flush=True)
        out[mode] = r
        del m
    out["greedy_identical"] = {str(b): bool(torch.equal(v[0], v[1])) for b, v in toks.items()}
    return out


def weight_bytes_str(n):
    return f"{n / 1e9:.2f} GB"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "w4_prefill_bench.json"))
    ap.add_argument("--skip-model", action="store_true")
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_w4_prefill needs the B200")
    res = dict(card=card(), torch=torch.__version__, note="synthetic group-128 codes, bf16; L2 not flushed between launches (weights "
                                                           "rotate over > 300 MB of copies)")
    res["projections"] = projections((64, 128, 576, 2464, 18432))
    if not args.skip_model:
        res["model"] = whole_model(args.steps)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
