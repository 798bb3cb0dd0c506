"""4-bit-only models (w4_only=True) on CPU: the mode equals the default GPTQ mode through the C-ABI double, every refusal raises,
gptq_w4_pack rejects linears that do not share one group size, and cts_gemm_w4_prefill's SOURCE runs on the CUDA-on-CPU shim bit for
bit like the shim's cts_gemm on the dequantised weight."""
import json

import numpy as np
import pytest
import torch

from chatts_b200 import ChatTSConfig, ChatTSProcessor, SimpleTokenizer
from chatts_b200.weights import pack_gptq_linear, synthetic_state_dict
from tests.w4_prefill_support import add_w4_prefill, shim_context_w4p

KW = dict(device="cpu", dtype=torch.bfloat16, max_seq_len=256, page_size=16, use_cuda_graph=False)


def _cfg(intermediate_size=768):
    return ChatTSConfig.tiny(intermediate_size=intermediate_size)       # 768: every K a multiple of 128 (fragment-major layout)


def _enc(cfg, batch):
    proc = ChatTSProcessor(SimpleTokenizer(cfg.ts_token_start_index, cfg.pad_token_id, cfg.eos_token_id), cfg)
    texts = ["A <ts><ts/> ?"] + [f"p{i} " + "w " * (i % 5) for i in range(1, batch)]
    return proc(text=texts, timeseries=[np.sin(np.arange(120) / 9) * 4], padding=True, return_tensors="pt")


def _models(cabi_double, max_batch=40, **kw):
    from chatts_b200.model import ChatTSForCausalLM
    add_w4_prefill(cabi_double)
    cabi_double.split = 2
    cfg = _cfg()
    sd = synthetic_state_dict(cfg, seed=3, device="cpu", std=0.05)
    md = ChatTSForCausalLM(cfg, sd, max_batch=max_batch, **KW, **kw).quantize_w4_synthetic(group_size=64)
    mo = ChatTSForCausalLM(cfg, sd, max_batch=max_batch, **KW, **kw).quantize_w4_synthetic(group_size=64, w4_only=True)
    return cfg, md, mo


def test_w4_only_mode_equals_the_default_gptq_mode(cabi_double):
    cfg, md, mo = _models(cabi_double)
    assert mo.w4_only and not md.w4_only
    assert all(w is None for lst in (mo.wqkv, mo.wo, mo.wgu, mo.wd) for w in lst)
    calls = []
    real = cabi_double.gemm_w4_prefill
    cabi_double.gemm_w4_prefill = lambda *a, **k: (calls.append(k.get("epilogue")), real(*a, **k))[1]
    for batch in (34, 2):                       # a 34-row decode batch takes the T > 32 path; 2 rows the decode kernel
        enc = _enc(cfg, batch)
        a, b = md(**enc, logits_to_keep=0).logits, mo(**enc, logits_to_keep=0).logits
        assert all(torch.equal(p, q) for p, q in zip(a, b))
        assert torch.equal(md.generate(**enc, max_new_tokens=6, ignore_eos=True), mo.generate(**enc, max_new_tokens=6, ignore_eos=True))
    assert calls and set(calls) <= {0, 3, 4, 6}


def test_w4_only_refusals(cabi_double, monkeypatch):
    from chatts_b200.model import ChatTSForCausalLM
    from chatts_b200.train import LoraTrainer
    cfg, md, mo = _models(cabi_double, max_batch=2)
    with pytest.raises(ValueError, match="w4_only"):
        mo.merge_lora({"model.layers.0.self_attn.q_proj.lora_A.weight": torch.zeros(4, 256),
                       "model.layers.0.self_attn.q_proj.lora_B.weight": torch.zeros(256, 4)})
    with pytest.raises(ValueError, match="w4_only"):
        LoraTrainer(mo)
    sd = synthetic_state_dict(cfg, seed=3, device="cpu", std=0.05)
    m = ChatTSForCausalLM(cfg, sd, max_batch=2, **KW)
    m.tp_size = 2
    with pytest.raises(ValueError):
        m.quantize_w4_synthetic(group_size=64, w4_only=True)
    with pytest.raises(ValueError, match="use_fused_decode"):
        ChatTSForCausalLM(cfg, sd, max_batch=2, use_fused_decode=1, **KW).quantize_w4_synthetic(group_size=64, w4_only=True)
    # the shapes only the row-layout tcgen05 decode kernel takes (a K of 704 is not a multiple of 128), or that kernel chosen explicitly
    cfg704 = _cfg(704)
    sd704 = synthetic_state_dict(cfg704, seed=3, device="cpu", std=0.05)
    with pytest.raises(ValueError, match="fragment-major"):
        ChatTSForCausalLM(cfg704, sd704, max_batch=2, **KW).quantize_w4_synthetic(group_size=64, w4_only=True)
    monkeypatch.setenv("CTS_W4_KERNEL", "tc5")
    with pytest.raises(ValueError, match="fragment-major"):
        ChatTSForCausalLM(cfg, sd, max_batch=2, **KW).quantize_w4_synthetic(group_size=64, w4_only=True)


def _gptq_dir(tmp_path, cfg, name, group, act_order=False, quant_group=None):
    from safetensors.torch import save_file
    sd = synthetic_state_dict(cfg, seed=9, device="cpu", std=0.05)
    out = {}
    for k, v in sd.items():
        if ".layers." in k and k.endswith("_proj.weight"):
            qw, qz, sc, gi = pack_gptq_linear(v.float(), group if group > 0 else v.shape[1], 1)
            if act_order:
                gi = gi.flip(0).contiguous()
            base = k[: -len(".weight")]
            out.update({base + ".qweight": qw, base + ".qzeros": qz, base + ".scales": sc, base + ".g_idx": gi})
        else:
            out[k] = v.contiguous()
    d = tmp_path / name
    d.mkdir()
    conf = cfg.to_dict()
    conf["quantization_config"] = {"bits": 4, "group_size": group if quant_group is None else quant_group, "quant_method": "gptq"}
    json.dump(conf, open(d / "config.json", "w"))
    save_file(out, str(d / "model.safetensors"))
    return str(d), out, conf["quantization_config"]


def test_checkpoint_loads_refuse_what_the_4bit_kernels_cannot_represent(cabi_double, tmp_path):
    from chatts_b200.model import ChatTSForCausalLM
    from chatts_b200.weights import gptq_w4_pack
    cfg = _cfg()
    kw = dict(device="cpu", torch_dtype="bfloat16", max_batch=2, max_seq_len=256, page_size=16, use_cuda_graph=False)
    # group_size -1: one group per input column -- q/k/v/o/gate/up have 256 inputs, down_proj 768: no single group size
    path, sd, qc = _gptq_dir(tmp_path, cfg, "per_column", -1)
    assert gptq_w4_pack(sd, qc) == (None, 0)
    with pytest.raises(ValueError, match="w4_only"):
        ChatTSForCausalLM.from_pretrained(path, w4_only=True, **kw)
    path, _, _ = _gptq_dir(tmp_path, cfg, "act_order", 64, act_order=True)
    with pytest.raises(ValueError, match="w4_only"):
        ChatTSForCausalLM.from_pretrained(path, w4_only=True, **kw)
    assert ChatTSForCausalLM.from_pretrained(path, **kw).w4 is None            # the default load keeps the dense weights, as before
    plain = tmp_path / "plain"
    plain.mkdir()
    from safetensors.torch import save_file
    save_file({k: v.contiguous() for k, v in synthetic_state_dict(cfg, seed=1, device="cpu").items()}, str(plain / "model.safetensors"))
    json.dump(cfg.to_dict(), open(plain / "config.json", "w"))
    with pytest.raises(ValueError, match="GPTQ"):
        ChatTSForCausalLM.from_pretrained(str(plain), w4_only=True, **kw)


def test_gptq_checkpoint_w4_only_load_matches_the_default_load(cabi_double, tmp_path):
    from chatts_b200.model import ChatTSForCausalLM
    add_w4_prefill(cabi_double)
    cfg = _cfg()
    path, _, _ = _gptq_dir(tmp_path, cfg, "ckpt", 128)
    kw = dict(device="cpu", torch_dtype="bfloat16", max_batch=34, max_seq_len=256, page_size=16, use_cuda_graph=False)
    md = ChatTSForCausalLM.from_pretrained(path, **kw)
    mo = ChatTSForCausalLM.from_pretrained(path, w4_only=True, **kw)
    assert mo.w4_only and mo.w4["group_size"] == 128 and mo.w4["kernel"] == "mma"
    enc = _enc(cfg, 34)
    assert torch.equal(md.generate(**enc, max_new_tokens=4, ignore_eos=True), mo.generate(**enc, max_new_tokens=4, ignore_eos=True))


@pytest.mark.parametrize("epi,t,split", [(3, 70, 3), (4, 300, 1), (6, 130, 1)])
def test_w4_prefill_kernel_source_on_the_cpu_shim(epi, t, split):
    """csrc/gemm_w4_persistent.cu compiled for the CUDA-on-CPU shim (tcgen05 / TMA / mbarrier emulation) against csrc/gemm_tcgen05.cu
    in the same build on the dequantised weight: bit-identical."""
    from chatts_b200.weights import dequantize_w4, repack_w4_mma
    c = shim_context_w4p()
    n, k, gs, dt = 256, 384, 128, torch.bfloat16
    g = torch.Generator().manual_seed(epi + t)
    qw = torch.randint(0, 256, (n, k // 2), generator=g, dtype=torch.uint8)
    sc = ((torch.rand(n, k // gs, generator=g) + 0.5) * 0.01).to(dt)
    zp = torch.randint(1, 17, (n, k // gs), generator=g, dtype=torch.uint8)
    qwf, szp = repack_w4_mma(qw, sc, zp, gs)
    w = dequantize_w4(qw, sc, zp, gs)
    x = (torch.randn(t, k, generator=g) * 0.5).to(dt)
    shape = (split, t, n) if epi == 3 else (t, n // 2 if epi == 6 else n)
    ref = torch.full(shape, -3.0, dtype=torch.float32 if epi == 3 else dt)
    if epi == 4:
        ref.copy_(torch.randn(t, n, generator=g).to(dt))
    got = ref.clone()
    c.gemm(x, w, ref, residual=ref if epi == 4 else None, epilogue=epi, split_k=split, t=t)
    c.gemm_w4_prefill(x, qwf, szp, n, gs, got, residual=got if epi == 4 else None, epilogue=epi, split_k=split, t=t)
    assert torch.equal(got, ref) and not torch.equal(got, torch.full_like(got, -3.0))
