"""cts_gemm_w4_prefill (csrc/gemm_w4_persistent.cu: persistent tcgen05 W4A16 GEMM over the fragment-major 4-bit copy) against cts_gemm on
the dequantised weight -- the same 16-bit operand values through the same 64-wide K blocks and K = 16 MMAs, so every epilogue and every
split must be BIT-IDENTICAL (torch.equal) -- its argument checks, and the 4-bit-only model mode (w4_only=True) built on it: prefill
logits, greedy tokens, memory, the GPTQ checkpoint load and the public surfaces."""
import ctypes as C
import gc

import numpy as np
import pytest
import torch

from tests.gpu_util import ctx, record

pytestmark = pytest.mark.gpu
NONE, PARTIAL, RES, IL = 0, 3, 4, 6
EPI_NAME = {NONE: "none", PARTIAL: "partial", RES: "res", IL: "swiglu_il"}

# (tag, n, k, group size, t, epilogue, split ("auto" = what the model's _splits picks), variant)
CASES = [
    # ChatTS-14B projections: qkv (7168 x 5120, bias), o (5120 x 5120), interleaved gate_up (27648 x 5120), down (5120 x 13824)
    ("14b", 7168, 5120, 128, 577, NONE, 1, "bias"),
    ("14b", 7168, 5120, 64, 2464, NONE, 1, "bias"),
    ("14b", 7168, 5120, 128, 33, NONE, 1, "bias"),
    ("14b", 7168, 5120, 128, 129, NONE, 1, ""),
    ("14b", 5120, 5120, 128, 577, RES, 1, ""),
    ("14b", 5120, 5120, 64, 18432, RES, 1, "alias"),
    ("14b", 5120, 13824, 128, 2464, RES, 1, "alias"),
    ("14b", 5120, 13824, 64, 128, RES, 1, "bias"),
    ("14b", 27648, 5120, 128, 577, IL, 1, ""),
    ("14b", 27648, 5120, 64, 129, IL, 1, ""),
    ("14b", 27648, 5120, 128, 18432, IL, 1, ""),
    ("14b", 7168, 5120, 128, 64, PARTIAL, 1, ""),
    ("14b", 7168, 5120, 128, 64, PARTIAL, 2, ""),
    ("14b", 7168, 5120, 128, 64, PARTIAL, "auto", ""),
    ("14b", 5120, 5120, 64, 33, PARTIAL, "auto", ""),
    ("14b", 27648, 5120, 128, 128, PARTIAL, "auto", ""),
    ("14b", 27648, 5120, 64, 64, PARTIAL, 2, ""),
    ("14b", 5120, 13824, 128, 128, PARTIAL, "auto", ""),
    ("14b", 5120, 13824, 64, 33, PARTIAL, 1, ""),
    ("14b", 5120, 5120, 128, 2464, PARTIAL, 1, ""),
    # odd shapes: n not a multiple of 256 (or of 128), t not a multiple of the 256-token tile, short K ranges
    ("small", 200, 768, 64, 5, NONE, 1, "bias"),
    ("small", 200, 768, 64, 129, RES, 1, "alias"),
    ("small", 136, 256, 128, 300, NONE, 1, ""),
    ("small", 384, 1024, 128, 577, IL, 1, ""),
    ("small", 640, 512, 64, 33, PARTIAL, 3, ""),
    ("small", 136, 256, 128, 300, PARTIAL, 4, ""),
    ("small", 328, 384, 128, 64, RES, 1, "bias"),
    ("small", 256, 512, 64, 130, PARTIAL, "auto", ""),
]


def _id(c):
    tag, n, k, gs, t, epi, split, var = c
    return f"{tag}-n{n}-k{k}-g{gs}-t{t}-{EPI_NAME[epi]}-s{split}" + (f"-{var}" if var else "")


_cache = {}


def _weights(n, k, gs, dtype):
    """Random codes / scales / zero points (seeded by the shape) -> (fragment-major qwf, szp, the dequantised dense weight) on the device."""
    from chatts_b200.weights import dequantize_w4, repack_w4_mma
    key = (n, k, gs, dtype)
    if key not in _cache:
        _cache.clear()
        g = torch.Generator().manual_seed(n * 7 + k + gs)
        qw = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8).cuda()
        sc = ((torch.rand(n, k // gs, generator=g) + 0.5) * 0.01).to(dtype).cuda()
        zp = torch.randint(1, 17, (n, k // gs), generator=g, dtype=torch.uint8).cuda()
        qwf, szp = repack_w4_mma(qw, sc, zp, gs)
        _cache[key] = (qwf.contiguous(), szp.contiguous(), dequantize_w4(qw, sc, zp, gs).contiguous())
    return _cache[key]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("case", CASES, ids=[_id(c) for c in CASES])
def test_w4_prefill_bit_identical_to_the_dense_gemm(case, dtype):
    _, n, k, gs, t, epi, split, var = case
    c = ctx()
    if split == "auto":      # the model's choice at this T (gate_up: the interleaved weight of n rows = 2 x intermediate)
        split = c.suggest_split(n // 2, k, t, True) if n == 27648 else c.suggest_split(n, k, t)
    qwf, szp, w = _weights(n, k, gs, dtype)
    g = torch.Generator().manual_seed(t + n)
    x = (torch.randn(t, k, generator=g) * 0.5).to(dtype).cuda()
    bias = (torch.randn(n, generator=g) * 0.1).to(dtype).cuda() if var == "bias" else None
    if epi == PARTIAL:
        ref = torch.full((split, t, n), -3.0, device="cuda")
    else:
        ref = torch.full((t, n // 2 if epi == IL else n), -3.0, device="cuda", dtype=dtype)
    resid = None
    if epi == RES:
        resid = (torch.randn(t, n, generator=g)).to(dtype).cuda()
        if var == "alias":
            ref.copy_(resid)
    got = ref.clone()
    kw = dict(bias=bias, epilogue=epi, split_k=split, t=t)
    c.gemm(x, w, ref, residual=(ref if var == "alias" else resid), **kw)
    c.gemm_w4_prefill(x, qwf, szp, n, gs, got, residual=(got if var == "alias" else resid), **kw)
    torch.cuda.synchronize()
    same = torch.equal(got, ref)
    record("gemm_w4_prefill", case=_id(case), dtype=str(dtype), split=split, bit_identical=int(same),
           max_abs_diff=0.0 if same else float((got.float() - ref.float()).abs().max()))
    assert same


def test_w4_prefill_bad_arguments_write_nothing():
    """Every precondition of cts_gemm_w4p_args returns CTS_ERR_BAD_ARG with a message, and nothing is launched: out keeps its bytes."""
    from chatts_b200 import _cabi
    c = ctx()
    n, k, gs, t = 256, 512, 128, 160
    dtype = torch.bfloat16
    qwf, szp, _ = _weights(n, k, gs, dtype)
    x = torch.randn(t, k, dtype=torch.float32).to(dtype).cuda()
    out = torch.full((t, n), 5.0, device="cuda", dtype=dtype)
    bias = torch.zeros(n, device="cuda", dtype=dtype)

    def args(**over):
        a = _cabi.GemmW4pArgs()
        a.qw, a.szp, a.x, a.out, a.bias, a.residual = qwf.data_ptr(), szp.data_ptr(), x.data_ptr(), out.data_ptr(), None, None
        a.n, a.k, a.t, a.x_ld, a.out_ld = n, k, t, k, n
        a.group_size, a.split_k, a.dtype, a.epilogue = gs, 1, _cabi.BF16, NONE
        for key, v in over.items():
            setattr(a, key, v)
        return a

    ok = args()
    assert c.lib.cts_gemm_w4_prefill(c.h, C.byref(ok), _cabi._stream()) == 0          # the baseline is valid
    torch.cuda.synchronize()
    out.fill_(5.0)
    bad = {
        "null qw": dict(qw=None), "null szp": dict(szp=None), "null x": dict(x=None), "null out": dict(out=None),
        "t = 0": dict(t=0), "n = 0": dict(n=0), "k % 128": dict(k=448, x_ld=448), "dtype": dict(dtype=7),
        "group 96": dict(group_size=96), "group 192": dict(group_size=192), "group 1024 > k": dict(group_size=1024),
        "split 0": dict(split_k=0), "split > k / 64": dict(split_k=9), "split with NONE": dict(split_k=2),
        "GELU": dict(epilogue=1), "SWIGLU": dict(epilogue=2), "SPLITK_F32": dict(epilogue=5),
        "RESIDUAL without residual": dict(epilogue=RES), "bias with PARTIAL": dict(epilogue=PARTIAL, bias=bias.data_ptr()),
        "bias with SWIGLU_IL": dict(epilogue=IL, bias=bias.data_ptr(), out_ld=n // 2),
        "x_ld < k": dict(x_ld=k - 8), "x_ld % 8": dict(x_ld=k + 4), "x misaligned": dict(x=x.data_ptr() + 2),
        "qw misaligned": dict(qw=qwf.data_ptr() + 8), "szp misaligned": dict(szp=szp.data_ptr() + 4),
        "out_ld < n": dict(out_ld=n - 1), "SWIGLU_IL out_ld < n / 2": dict(epilogue=IL, out_ld=n // 2 - 1),
        "SWIGLU_IL t <= 128": dict(epilogue=IL, t=128, out_ld=n // 2), "SWIGLU_IL n % 128": dict(epilogue=IL, n=192, out_ld=96),
    }
    for name, over in bad.items():
        a = args(**over)
        rc = c.lib.cts_gemm_w4_prefill(c.h, C.byref(a), _cabi._stream())
        msg = c.lib.cts_last_error(c.h)
        assert rc == -1, name
        assert msg, name
    assert c.lib.cts_gemm_w4_prefill(None, C.byref(ok), _cabi._stream()) == -1
    torch.cuda.synchronize()
    assert bool((out == 5.0).all())


# ------------------------------------------------------------------------------------------------------------------------------ model
def _tiny(qwen3):
    from chatts_b200 import ChatTSConfig
    from chatts_b200.weights import synthetic_state_dict
    cfg = ChatTSConfig.tiny(intermediate_size=768)          # every K a multiple of 128: the fragment-major layout
    if qwen3:
        cfg.qk_norm, cfg.attention_bias = True, False
    return cfg, synthetic_state_dict(cfg, seed=5, device="cpu", dtype=torch.bfloat16, std=0.05)


def _prompts(cfg, batch):
    from chatts_b200 import ChatTSProcessor, SimpleTokenizer
    proc = ChatTSProcessor(SimpleTokenizer(cfg.ts_token_start_index, cfg.pad_token_id, cfg.eos_token_id), cfg)
    x = np.arange(200)
    texts = ["A <ts><ts/> ?"] + [f"prompt {i}: " + "some words " * (i % 9) for i in range(1, batch)]
    return proc(text=texts, timeseries=[np.sin(x / 9) * 4], padding=True, return_tensors="pt")


@pytest.mark.parametrize("qwen3", [False, True], ids=["qwen2", "qwen3"])
def test_model_w4_only_matches_the_default_gptq_mode(qwen3):
    """The same seeds, quantize_w4_synthetic(group_size=64) with and without w4_only: the default mode runs prefill and 33-128-row
    decode steps on the dense dequantised copy, the 4-bit-only mode on cts_gemm_w4_prefill with the same epilogues and splits, so
    prefill logits and greedy tokens must be IDENTICAL -- at a decode batch of 40 rows (the 33-128-row path) and of 2 (T <= 32)."""
    from chatts_b200.model import ChatTSForCausalLM
    cfg, sd = _tiny(qwen3)
    kw = dict(dtype=torch.bfloat16, max_batch=48, max_seq_len=256, page_size=16)
    md = ChatTSForCausalLM(cfg, sd, **kw).quantize_w4_synthetic(group_size=64)
    mo = ChatTSForCausalLM(cfg, sd, **kw).quantize_w4_synthetic(group_size=64, w4_only=True)
    assert mo.w4_only and all(w is None for lst in (mo.wqkv, mo.wo, mo.wgu, mo.wd) for w in lst)
    for batch in (40, 2):
        enc = _prompts(cfg, batch)
        a, b = md(**enc, logits_to_keep=0).logits, mo(**enc, logits_to_keep=0).logits
        assert all(torch.equal(p, q) for p, q in zip(a, b))
        l0 = mo.ctx.launches
        ta = md.generate(**enc, max_new_tokens=16, ignore_eos=True)
        tb = mo.generate(**enc, max_new_tokens=16, ignore_eos=True)
        assert mo.ctx.launches > l0
        record("w4_only_model", qwen3=int(qwen3), batch=batch, tokens_identical=int(torch.equal(ta, tb)), prefill_T=int(enc["attention_mask"].sum()))
        assert torch.equal(ta, tb)


def test_model_w4_only_frees_the_dense_projections():
    from chatts_b200.model import ChatTSForCausalLM
    cfg, sd = _tiny(False)
    kw = dict(dtype=torch.bfloat16, max_batch=4, max_seq_len=256, page_size=16)
    gc.collect()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    md = ChatTSForCausalLM(cfg, sd, **kw).quantize_w4_synthetic(group_size=128)
    dense = sum(w.numel() * w.element_size() for lst in (md.wqkv, md.wo, md.wgu, md.wd) for w in lst)
    gc.collect()
    torch.cuda.synchronize()
    a_default = torch.cuda.memory_allocated() - base
    del md
    gc.collect()
    mo = ChatTSForCausalLM(cfg, sd, **kw).quantize_w4_synthetic(group_size=128, w4_only=True)
    gc.collect()
    torch.cuda.synchronize()
    a_only = torch.cuda.memory_allocated() - base
    record("w4_only_memory", default_bytes=a_default, w4_only_bytes=a_only, dense_projection_bytes=dense)
    assert a_default - a_only >= dense
    assert all(w is None for lst in (mo.wqkv, mo.wo, mo.wgu, mo.wd) for w in lst)


def _gptq_dir(tmp_path, group=128):
    import json
    from safetensors.torch import save_file
    from chatts_b200 import ChatTSConfig
    from chatts_b200.weights import pack_gptq_linear, synthetic_state_dict
    cfg = ChatTSConfig.tiny(intermediate_size=768)
    sd = synthetic_state_dict(cfg, seed=9, device="cpu", dtype=torch.bfloat16, std=0.05)
    out = {}
    for k, v in sd.items():
        if ".layers." in k and k.endswith("_proj.weight"):
            qw, qz, sc, gi = pack_gptq_linear(v.float(), group, 1)
            base = k[: -len(".weight")]
            out.update({base + ".qweight": qw, base + ".qzeros": qz, base + ".scales": sc, base + ".g_idx": gi})
        else:
            out[k] = v.contiguous()
    d = tmp_path / "ckpt"
    d.mkdir()
    conf = cfg.to_dict()
    conf["quantization_config"] = {"bits": 4, "group_size": group, "quant_method": "gptq"}
    json.dump(conf, open(d / "config.json", "w"))
    save_file(out, str(d / "model.safetensors"))
    return cfg, str(d)


def test_gptq_checkpoint_w4_only_load_matches_the_default_load(tmp_path):
    from chatts_b200.model import ChatTSForCausalLM
    cfg, path = _gptq_dir(tmp_path)
    kw = dict(torch_dtype="bfloat16", max_batch=40, max_seq_len=256, page_size=16)
    md = ChatTSForCausalLM.from_pretrained(path, **kw)
    mo = ChatTSForCausalLM.from_pretrained(path, w4_only=True, **kw)
    assert md.w4 is not None and not md.w4_only and mo.w4_only and mo.w4["group_size"] == 128
    assert all(w is None for lst in (mo.wqkv, mo.wo, mo.wgu, mo.wd) for w in lst)
    for batch in (2, 36):
        enc = _prompts(cfg, batch)
        ta = md.generate(**enc, max_new_tokens=12, ignore_eos=True)
        tb = mo.generate(**enc, max_new_tokens=12, ignore_eos=True)
        record("w4_only_gptq_checkpoint", batch=batch, tokens_identical=int(torch.equal(ta, tb)))
        assert torch.equal(ta, tb)


def test_w4_only_public_surfaces(tmp_path):
    """LLM(model=path, w4_only=True).generate(...) and one request through the continuous engine complete."""
    from chatts_b200.engine import ContinuousEngine
    from chatts_b200.vllm_compat import LLM, SamplingParams
    cfg, path = _gptq_dir(tmp_path)
    llm = LLM(model=path, w4_only=True, max_model_len=256, max_num_seqs=4)
    assert llm.model.w4_only
    outs = llm.generate(["hello there", "a second prompt"], SamplingParams(max_tokens=6, ignore_eos=True))
    assert len(outs) == 2 and all(len(o.outputs[0].token_ids) == 6 for o in outs)
    enc = _prompts(cfg, 1)
    eng = ContinuousEngine(llm.model, slots=4, steps_per_round=3, max_prefill_batch=1)
    eng.add_request(enc["input_ids"][0], enc["timeseries"], max_new_tokens=5, ignore_eos=True)
    done = eng.run()
    eng.close()
    assert len(done) == 1 and len(done[0].tokens) == 5
