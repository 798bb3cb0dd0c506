"""ChatTSForCausalLM on B200: TS encoder -> merge at ``<ts>`` -> Qwen2 decoder -> lm_head, behind the
``generate()`` surface the reference's callers use (README.md:88-103, demo/demo_hf.ipynb cells 3-5,
chatts/utils/inference_tsmllm_deepspeed.py:89-106).

Replaces, for this path only: the checkpoint's remote-code ``Qwen2TSForCausalLM`` (HF surface) and
``chatts.vllm.chatts_vllm.Qwen2TSForCausalLM`` (chatts_vllm.py:452-625).  All arithmetic runs in the sm_100a
kernels of libchatts_b200.so; torch provides device memory, streams, CUDA-graph capture and
torch.distributed.  There is no CPU or eager-torch fallback: constructing the model without a B200 raises.

Decode is a single CUDA graph per batch size: embedding gather -> [split-K tcgen05 GEMM -> fused
reduce(+bias+RoPE+KV write | +residual+RMSNorm | SwiGLU)] x layers -> paged flash-decode -> lm_head -> argmax
-> device-side advance (next id, position, KV slot), so a step replays with no host round trip.
"""
import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _cabi, layout
from .trace import span
from ._cabi import EPI_NONE, EPI_PARTIAL_F32, EPI_RESIDUAL, EPI_SWIGLU_IL
from .config import ChatTSConfig
from .ts_encoder import TimeSeriesEmbedding
from .weights import load_checkpoint, shard_tensor, synthetic_state_dict


@dataclass
class CausalLMOutput:
    logits: torch.Tensor


def rope_tables(cfg, n_pos, dtype, device):
    """cos/sin exactly as transformers computes them (modeling_qwen2.py:88-113): fp32 inv_freq, fp32 outer
    product, fp32 cos/sin, THEN cast to the model dtype.  Computed once on the host at load time (not on the
    hot path) so the table is bit-identical to the reference's; [n_pos, head_dim/2] because emb = cat(f, f)."""
    d = cfg.head_dim
    inv_freq = 1.0 / (float(cfg.rope_theta) ** (torch.arange(0, d, 2, dtype=torch.int64).to(torch.float32) / d))
    pos = torch.arange(n_pos, dtype=torch.float32)
    freqs = (inv_freq[:, None] @ pos[None, :]).transpose(0, 1)
    return freqs.cos().to(dtype).to(device).contiguous(), freqs.sin().to(dtype).to(device).contiguous()


class PagePool:
    """Free-list allocator over the pages of the KV cache ([num_pages, nkv, page_size, d] per layer and K/V)."""

    def __init__(self, num_pages):
        self.free = list(range(num_pages - 1, -1, -1))
        self.num_pages = num_pages

    def alloc(self, n):
        if n > len(self.free):
            raise RuntimeError(f"KV cache exhausted: need {n} pages, {len(self.free)} free of {self.num_pages}")
        return [self.free.pop() for _ in range(n)]

    def release(self, pages):
        self.free.extend(reversed(pages))


class _Step:
    """Static buffers of one decode configuration (batch size) + its captured CUDA graphs."""
    pass


class ChatTSForCausalLM:
    def __init__(self, config, state_dict, device="cuda", dtype=torch.bfloat16, tp_rank=0, tp_size=1,
                 max_batch=32, max_seq_len=2048, page_size=64, use_cuda_graph=True, comm=None,
                 use_peer_allreduce=True, graph_with_tp=True, use_chain=None, use_sample_kernel=None, use_native_step=None, use_fused_decode=None, use_peer_ll=None, dense_projections=True):
        """dense_projections=False: the decoder projections (q/k/v/o/gate/up/down weights) are not loaded from ``state_dict``; the
        model is unusable until attach_w4(..., w4_only=True) supplies them as 4-bit weights (from_pretrained(path, w4_only=True))."""
        if not torch.cuda.is_available():
            raise _cabi.CtsError("chatts_b200 needs a B200 (sm_100a) GPU; there is no CPU fallback")
        self.config, self.dtype = config, dtype
        self.device = torch.device(device if str(device) != "cuda" else f"cuda:{torch.cuda.current_device()}")
        self.tp_rank, self.tp_size, self.comm = tp_rank, tp_size, comm
        self.ctx = _cabi.get_context(self.device)
        cfg = config
        assert cfg.num_key_value_heads % tp_size == 0 and cfg.num_attention_heads % tp_size == 0
        self.nh, self.nkv, self.d = cfg.num_attention_heads // tp_size, cfg.num_key_value_heads // tp_size, cfg.head_dim
        self.H, self.I = cfg.hidden_size, cfg.intermediate_size // tp_size
        self.n_qkv = (self.nh + 2 * self.nkv) * self.d             # fused q|k|v output features (per rank)
        self.V = cfg.vocab_size // tp_size if tp_size > 1 else cfg.vocab_size
        self.L = cfg.num_hidden_layers
        self.eps = float(cfg.rms_norm_eps)
        self.page_size, self.max_batch, self.max_seq_len = page_size, max_batch, max_seq_len
        self.max_pages = (max_seq_len + page_size - 1) // page_size
        self.use_cuda_graph = use_cuda_graph
        self.graph_with_tp = graph_with_tp
        import os as _os
        self.use_chain = bool(int(_os.environ.get("CTS_DECODE_CHAIN", "0"))) if use_chain is None else bool(use_chain)
        # the whole decode step enqueued by one C call (cts_decoder_step) instead of ~440 ctypes calls: identical launches; off by
        # default until compared with the Python orchestration on a B200 (CTS_NATIVE_STEP=1 / use_native_step=True)
        self.use_native_step = bool(int(_os.environ.get("CTS_NATIVE_STEP", "0"))) if use_native_step is None else bool(use_native_step)
        # decode GEMMs with the split-K reduction and the projection tail fused in through a thread-block cluster
        # (csrc/gemm_decode_fused.cu: 9 -> 7 dependent stages per layer); off by default until it has run on a B200
        #   1: projections fused with their tails, plain RMSNorm launches between them (7 stages, bit-identical to the default path)
        #   2: the RMSNorms too -- the residual projections emit per-tile sums of squares, the next projection builds its normalised
        #      token operand itself (5 stages; single GPU only)
        self.use_fused_decode = int(_os.environ.get("CTS_DECODE_FUSED", "0")) if use_fused_decode is None else int(use_fused_decode)
        # tensor parallelism: low-latency two-shot all-reduce (cts_peer_allreduce_ll) instead of the one-shot push kernel
        # (default since round 2: validated across 2 B200s -- same logits, same tokens on every rank -- and 19-25 % faster per step
        #  than the one-shot kernel at TP2, profiles/r2_tp2_variants.txt; CTS_PEER_LL=0 selects the one-shot kernel)
        self.use_peer_ll = (_os.environ.get("CTS_PEER_LL", "1") == "1") if use_peer_ll is None else bool(use_peer_ll)
        # row-parallel exchange of prefill-sized steps: "rs_ag" (default: fp32 reduce-scatter + 16-bit all-gather of the result), "fp32"
        # (one fp32 all-reduce, rounds 1-2), "16bit" (all-reduce in the model dtype: vLLM's semantics, fastest, re-rounds the running sum)
        self.tp_prefill_exchange = _os.environ.get("CTS_TP_PREFILL_EXCHANGE", "rs_ag")
        self._nccl = False
        if tp_size > 1 and torch.distributed.is_available() and torch.distributed.is_initialized():
            try:
                self._nccl = str(torch.distributed.get_backend(comm)) == "nccl"   # comm None = the default group; gloo (CPU tests) has no reduce_scatter: fp32 all-reduce there
            except Exception:
                self._nccl = False
        # sampled decoding through cts_sample_advance (csrc/sampling.cu): temperature / top-k / top-p / multinomial / advance in ONE
        # launch per step, no torch op on the path (validated on a B200: 17 cases against the CPU statement that is itself checked
        # against transformers' logits warpers).  Default since round 2; CTS_SAMPLE_KERNEL=0 selects the torch-op fallback.
        self.use_sample_kernel = bool(int(_os.environ.get("CTS_SAMPLE_KERNEL", "1"))) if use_sample_kernel is None else bool(use_sample_kernel)
        # bytes of the NEXT GEMM's weight a decode GEMM prefetches into L2 once its own stream is requested.  OFF by default: measured
        # on a B200 (profiles/r2_next_prefetch_ab.txt) it fills the gaps between the weight streams but makes the step SLOWER
        # (b=32: 6.59 ms without, 6.83 / 7.00 / 7.08 ms with 24 / 48 / 80 MB) -- the prefetched lines do not survive the current
        # GEMM's stream through L2, so the bytes are read twice.  CTS_NEXT_PREFETCH_MB=<n> turns it on for experiments.
        self.next_prefetch_bytes = int(float(_os.environ.get("CTS_NEXT_PREFETCH_MB", "0")) * (1 << 20))
        self.w4 = None               # W4A16 decode weights (csrc/gemm_w4.cu): set by attach_w4 / quantize_w4_synthetic / from_pretrained(GPTQ)
        self.w4_only = False         # True: the 4-bit copy is the ONLY copy of the projections (attach_w4(..., w4_only=True))
        self._load(state_dict, dense_projections)
        # every position the page table can address has a row in the rotary tables (max_pages * page_size >= max_seq_len), capped by
        # the model's max_position_embeddings; _alloc_pages rejects sequences beyond it (no silent out-of-bounds cos/sin read)
        n_pos = min(cfg.max_position_embeddings, max(self.max_pages * page_size, 16))
        self.cos, self.sin = rope_tables(cfg, n_pos, dtype, self.device)
        self.n_pos = n_pos
        num_pages = max_batch * self.max_pages
        self.kv = torch.zeros(self.L, 2, num_pages, self.nkv, page_size, self.d, device=self.device, dtype=dtype)
        self.pool = PagePool(num_pages)
        self._steps = {}
        self.peer, self.peer_tokens = None, 0
        if tp_size > 1 and use_peer_allreduce:
            from .tp import PeerBuffers
            self.peer_tokens = max(max_batch, 64)
            self.peer = PeerBuffers(self.ctx, tp_rank, tp_size, self.peer_tokens, self.H, group=comm)

    # ------------------------------------------------------------------------------------------ loading
    def _load(self, sd, dense_projections=True):
        cfg, dev, dt = self.config, self.device, self.dtype

        def take(name):
            t = sd[name]
            t = shard_tensor(name, t, cfg, self.tp_rank, self.tp_size)
            return t.to(dev, dt).contiguous()

        self.embed = take("model.embed_tokens.weight")
        self.final_norm = take("model.norm.weight")
        self.lm_head = take("lm_head.weight") if "lm_head.weight" in sd else (
            shard_tensor("lm_head.weight", sd["model.embed_tokens.weight"], cfg, self.tp_rank, self.tp_size).to(dev, dt).contiguous())
        self.ln1, self.ln2, self.wqkv, self.bqkv, self.wo, self.wgu, self.wd = [], [], [], [], [], [], []
        self.qn, self.kn = [], []
        for l in range(self.L):
            p = f"model.layers.{l}."
            self.ln1.append(take(p + "input_layernorm.weight"))
            self.ln2.append(take(p + "post_attention_layernorm.weight"))
            if (p + "self_attn.q_proj.bias") in sd:
                self.bqkv.append(torch.cat([take(p + f"self_attn.{n}_proj.bias") for n in "qkv"], 0).contiguous())
            else:
                self.bqkv.append(None)
            has_qkn = (p + "self_attn.q_norm.weight") in sd          # Qwen3 / ChatTS-8B
            self.qn.append(take(p + "self_attn.q_norm.weight") if has_qkn else None)
            self.kn.append(take(p + "self_attn.k_norm.weight") if has_qkn else None)
            if not dense_projections:
                for lst in (self.wqkv, self.wo, self.wgu, self.wd):
                    lst.append(None)
                continue
            self.wqkv.append(torch.cat([take(p + f"self_attn.{n}_proj.weight") for n in "qkv"], 0).contiguous())
            self.wo.append(take(p + "self_attn.o_proj.weight"))
            # gate/up INTERLEAVED per 128-row tile (64 gate rows, then the 64 matching up rows): SwiGLU becomes local to
            # one MMA tile (CTS_EPI_SWIGLU_IL in the persistent prefill GEMM; cts_reduce_swiglu(interleaved) at decode)
            g, u = take(p + "mlp.gate_proj.weight"), take(p + "mlp.up_proj.weight")
            assert g.shape[0] % 64 == 0, "intermediate_size (per rank) must be a multiple of 64"
            self.wgu.append(torch.stack([g.view(-1, 64, g.shape[1]), u.view(-1, 64, u.shape[1])], 1).reshape(2 * g.shape[0], g.shape[1]).contiguous())
            del g, u
            self.wd.append(take(p + "mlp.down_proj.weight"))
        ts_w = {k: v for k, v in sd.items() if k.startswith("ts_encoder.")}
        self.ts_encoder = TimeSeriesEmbedding(cfg.ts, ts_w, device=dev, dtype=dt) if ts_w else None

    @classmethod
    def from_synthetic(cls, config=None, seed=1234, device="cuda", dtype=torch.bfloat16, gen_device=None, **kw):
        """Random-init weights at the config's shapes (no checkpoint exists offline).  ``gen_device='cpu'`` gives
        values identical to the CPU oracle's; the default generates on the GPU (14B in seconds)."""
        config = config or ChatTSConfig.chatts_14b()
        sd = synthetic_state_dict(config, seed=seed, device=gen_device or device, dtype=dtype)
        return cls(config, sd, device=device, dtype=dtype, **kw)

    @classmethod
    def from_pretrained(cls, path, device_map=None, torch_dtype=None, trust_remote_code=True, device=None, w4_only=False, **kw):
        """AutoModelForCausalLM.from_pretrained surface (README.md:88): config.json + safetensors shards.
        w4_only=True (GPTQ-Int4 checkpoints): the decoder projections are never dequantised; the 4-bit copy is their only copy and serves
        every step size (attach_w4).  A checkpoint the 4-bit kernels cannot represent raises ValueError instead of loading dense."""
        cfg = ChatTSConfig.from_json(path)
        dt = {"float16": torch.float16, "bfloat16": torch.bfloat16, torch.float16: torch.float16,
              torch.bfloat16: torch.bfloat16, None: getattr(torch, cfg.torch_dtype, torch.bfloat16)}[torch_dtype]
        dev = device if device is not None else (f"cuda:{device_map}" if isinstance(device_map, int) else (device_map or "cuda"))
        sd = load_checkpoint(path, device="cpu")
        w4_packed, w4_gs = None, 0
        if w4_only and not any(k.endswith(".qweight") for k in sd):
            raise ValueError("w4_only=True needs a GPTQ-Int4 checkpoint (no *.qweight tensors found)")
        if any(k.endswith(".qweight") for k in sd):                # GPTQ-Int4 checkpoint (README.md:52,262-263)
            import json as _json
            import os as _os
            from .weights import dequantize_gptq, gptq_w4_pack
            cj = _os.path.join(path, "config.json") if _os.path.isdir(path) else path
            qc = _json.load(open(cj)).get("quantization_config", {})
            # decode streams the 4-bit codes (csrc/gemm_w4.cu); prefill runs on a dequantised copy holding the same values (the scales
            # rounded to the model dtype, which is what the kernel multiplies with).  Act-order checkpoints, tensor parallelism and
            # CTS_W4=0 keep the dequantised weights only.
            if w4_only and (kw.get("tp_size", 1) != 1 or _os.environ.get("CTS_W4", "1") == "0"):
                raise ValueError("w4_only=True is single-GPU and needs the 4-bit kernels (tp_size=1, CTS_W4 not 0)")
            if _os.environ.get("CTS_W4", "1") != "0" and kw.get("tp_size", 1) == 1:
                w4_packed, w4_gs = gptq_w4_pack(sd, qc, dtype=dt)
            if w4_only:
                if w4_packed is None:
                    raise ValueError("w4_only=True: this GPTQ checkpoint cannot be represented by the 4-bit kernels (act-order g_idx, "
                                     "a group size that is not a multiple of 64 or differs between projections, or not 4-bit)")
                # the packed decoder projections never become dense; other quantised tensors (if any) are dequantised as before
                sd = {k: t for k, t in sd.items() if not (k.rsplit(".", 1)[0] in w4_packed and k.rsplit(".", 1)[1] in ("qweight", "qzeros", "scales", "g_idx"))}
            sd = dequantize_gptq(sd, qc, dtype=dt, scale_dtype=dt if w4_packed is not None else None)
        model = cls(cfg, sd, device=dev, dtype=dt, dense_projections=not w4_only, **kw)
        if w4_packed is not None:
            model.attach_w4(w4_packed, w4_gs, w4_only=w4_only)
        # generation_config.json: the defaults HF's generate() applies when the caller passes none (README.md:102 calls
        # model.generate(**inputs, max_new_tokens=300) with no sampling arguments)
        import json as _json2
        import os as _os2
        gc = _os2.path.join(path, "generation_config.json") if _os2.path.isdir(path) else ""
        if gc and _os2.path.exists(gc):
            model.generation_defaults = {k: v for k, v in _json2.load(open(gc)).items()
                                         if k in ("do_sample", "temperature", "top_p", "top_k", "eos_token_id", "pad_token_id", "max_new_tokens",
                                                  "repetition_penalty")}
        return model

    # ------------------------------------------------------------------------------------------ LoRA
    def merge_lora(self, adapter, lora_alpha=None, r=None):
        """PeftModel.from_pretrained(model, adapter).merge_and_unload() (demo/demo_lora.ipynb cells 3-4): fold LoRA adapters
        into the resident weights, W += (alpha / r) * B @ A, for q/k/v/o/gate/up/down_proj.  ``adapter`` is a directory with
        adapter_model.safetensors + adapter_config.json, or a name->tensor dict (PEFT names:
        ``...layers.{i}.self_attn.q_proj.lora_A.weight`` [r, in], ``...lora_B.weight`` [out, r]).  Load-time host logic:
        the merged weights then run through the same kernels."""
        import json
        import os
        import re
        if self.w4_only:
            raise ValueError("merge_lora needs the dense projection weights: this model keeps its projections as 4-bit weights only (w4_only)")
        if isinstance(adapter, str):
            cfg_path = os.path.join(adapter, "adapter_config.json")
            if os.path.exists(cfg_path):
                ac = json.load(open(cfg_path))
                lora_alpha = ac.get("lora_alpha", lora_alpha) if lora_alpha is None else lora_alpha
                r = ac.get("r", r) if r is None else r
            from safetensors.torch import load_file
            sd = load_file(os.path.join(adapter, "adapter_model.safetensors"))
        else:
            sd = dict(adapter)
        pairs = {}
        for name, t in sd.items():
            m = re.search(r"layers\.(\d+)\.(?:self_attn|mlp)\.(\w+_proj)\.lora_([AB])(?:\.\w+)?\.weight$", name)
            if m:
                pairs.setdefault((int(m.group(1)), m.group(2)), {})[m.group(3)] = t
        if not pairs:
            raise ValueError("no LoRA tensors (…{q,k,v,o,gate,up,down}_proj.lora_{A,B}.weight) found in the adapter")
        cfg, d = self.config, self.d
        nh_t, nkv_t = cfg.num_attention_heads, cfg.num_key_value_heads
        merged = 0
        for (l, proj), ab in sorted(pairs.items()):
            A, B = ab["A"].to(self.device, torch.float32), ab["B"].to(self.device, torch.float32)
            rank = A.shape[0]
            scale = float(lora_alpha if lora_alpha is not None else rank) / float(r if r is not None else rank)
            delta = (B @ A) * scale                                   # [out, in] in the unsharded HF shape
            delta = shard_tensor(f"model.layers.{l}.{'self_attn' if proj[0] in 'qkvo' else 'mlp'}.{proj}.weight", delta, cfg,
                                 self.tp_rank, self.tp_size)

            def add(w_rows, dlt):
                w_rows.copy_((w_rows.float() + dlt).to(self.dtype))

            if proj == "q_proj":
                add(self.wqkv[l][: self.nh * d], delta)
            elif proj == "k_proj":
                add(self.wqkv[l][self.nh * d:(self.nh + self.nkv) * d], delta)
            elif proj == "v_proj":
                add(self.wqkv[l][(self.nh + self.nkv) * d:], delta)
            elif proj == "o_proj":
                add(self.wo[l], delta)
            elif proj == "down_proj":
                add(self.wd[l], delta)
            elif proj in ("gate_proj", "up_proj"):
                # interleaved layout: tile k holds gate rows [64k, 64k+64) then up rows [64k, 64k+64)
                v = self.wgu[l].view(-1, 2, 64, self.H)
                sel = v[:, 0 if proj == "gate_proj" else 1]
                sel.copy_((sel.float() + delta.view(-1, 64, self.H)).to(self.dtype))
            else:
                continue
            merged += 1
        return merged          # in-place update: captured decode graphs keep reading the same (now merged) buffers

    # ------------------------------------------------------------------------------------------ W4A16 (GPTQ-Int4, README.md:52,262-263)
    def attach_w4(self, packed, group_size, w4_only=False):
        """Switch the DECODE step to the 4-bit weight stream.  ``packed``: {HF linear name (e.g. 'model.layers.3.mlp.up_proj'):
        (qw uint8 [out, in/2], scales [out, in/g], zeros uint8 [out, in/g])} in the layout of weights.py:repack_gptq_w4, for all
        seven projections of every layer.  The dense weights stay (prefill and every T > 32 step use them): they must hold the SAME
        values, i.e. weights.py:dequantize_gptq(..., scale_dtype=model dtype) -- 180 GB of HBM keep both copies.  Fused operands
        are assembled exactly like the dense ones: q|k|v stacked, gate/up interleaved per 64 rows.  Single GPU (a tensor-parallel
        row split would cut groups: down_proj's 13824 / 8 = 1728 inputs are not a multiple of the group size).
        w4_only=True: the 4-bit copy becomes the ONLY copy of the projections -- the dense wqkv / wo / wgu / wd are freed and every step
        size runs from the fragment-major codes (T <= 32 decode: cts_gemm_w4_mma; everything else: cts_gemm_w4_prefill with the epilogue
        and split factor the dense path uses, bit-identical to it).  Refused for shapes the fragment-major kernels cannot take, with the
        fused decode (use_fused_decode), and later by merge_lora and train.LoraTrainer, which need dense weights."""
        if self.tp_size != 1:
            raise ValueError("W4A16 decode weights are single-GPU (tensor parallelism uses the dequantised weights)")
        if w4_only and self.use_fused_decode:
            raise ValueError("w4_only=True: the fused decode GEMMs (use_fused_decode) read dense weights; build the model with use_fused_decode=0")
        dev = self.device
        gs = int(group_size)
        w4 = dict(group_size=gs, qkv=[], o=[], gu=[], d=[])

        def get(name):
            qw, sc, zp = packed[name]
            return qw.to(dev).contiguous(), sc.to(dev, self.dtype).contiguous(), zp.to(dev).contiguous()

        def il(a, b):                     # gate/up interleaved per 64 output rows, as _load does for the dense weight
            return torch.stack([a.view(-1, 64, a.shape[1]), b.view(-1, 64, b.shape[1])], 1).reshape(2 * a.shape[0], a.shape[1]).contiguous()

        for l in range(self.L):
            p = f"model.layers.{l}."
            q, k, v = (get(p + f"self_attn.{n}_proj") for n in "qkv")
            w4["qkv"].append(tuple(torch.cat([a, b, c], 0).contiguous() for a, b, c in zip(q, k, v)))
            w4["o"].append(get(p + "self_attn.o_proj"))
            g, u = get(p + "mlp.gate_proj"), get(p + "mlp.up_proj")
            w4["gu"].append(tuple(il(a, b) for a, b in zip(g, u)))
            w4["d"].append(get(p + "mlp.down_proj"))
        c = self.ctx
        import os as _os
        # kernel of the decode step: "mma" (default) = csrc/gemm_w4_mma.cu, the codes dequantised in registers from the fragment-major copy
        # built here (the row layout is dropped per layer once it is converted); "tc5" = csrc/gemm_w4.cu (tcgen05, bit-identical to the
        # dense GEMM, no faster than it: kept as the checker)
        w4["kernel"] = _os.environ.get("CTS_W4_KERNEL", "mma")
        k_dims = (self.H, self.nh * self.d, self.I)
        mma_ok = all(kd % 128 == 0 for kd in k_dims) and (gs == 64 or gs % 128 == 0)
        if w4_only and not (mma_ok and w4["kernel"] == "mma"):
            raise ValueError(f"w4_only=True needs the fragment-major 4-bit layout: every K ({k_dims}) a multiple of 128, group size 64 or a "
                             f"multiple of 128 (got {gs}), and CTS_W4_KERNEL=mma")
        if w4["kernel"] == "mma" and not mma_ok:
            w4["kernel"] = "tc5"          # the mma kernel's pipeline stage is 128 K wide (cts_gemm_w4f_args): odd shapes take the tcgen05 kernel
        if w4["kernel"] == "mma":
            from .weights import repack_w4_mma
            for kind in ("qkv", "o", "gu", "d"):
                for l in range(self.L):
                    qw, sc, zp = w4[kind][l]
                    w4[kind][l] = repack_w4_mma(qw, sc, zp, gs) + (int(qw.shape[0]),)
            w4["splits"] = None           # per batch size: _w4_splits
        else:
            w4["splits"] = dict(qkv=c.gemm_w4_suggest_split(self.n_qkv, self.H), o=c.gemm_w4_suggest_split(self.H, self.nh * self.d),
                                gu=c.gemm_w4_suggest_split(2 * self.I, self.H), d=c.gemm_w4_suggest_split(self.H, self.I))
        w4["only"] = bool(w4_only)
        self.w4 = w4
        if w4_only:
            # no dense copy: nothing may reach for one (None fails loudly), and no GEMM names a dense weight as its L2-prefetch successor
            for lst in (self.wqkv, self.wo, self.wgu, self.wd):
                lst[:] = [None] * self.L
            self.w4_only = True
            self.next_prefetch_bytes = 0
            self.__dict__.pop("_layer_list", None)          # the native step's cached operand list would keep the dense weights alive
        self._steps = {}                  # decode states (workspaces, captured graphs) are rebuilt for the new launches
        return self

    def quantize_w4_synthetic(self, group_size=128, seed=7, w4_only=False):
        """Benchmark / test helper (no GPTQ checkpoint exists offline): draw random 4-bit codes, scales and zero points at the model's
        shapes, REPLACE the dense weights by their dequantised values and attach the packed copy -- a W4A16 model whose prefill and
        decode paths see the same weights.  w4_only=True: the same codes (same seed), attached as the only copy (attach_w4)."""
        from .weights import dequantize_w4, W4_NIBBLE_OF_K  # noqa: F401
        g = torch.Generator(device=self.device).manual_seed(seed)
        packed = {}

        def make(n_out, n_in):
            qw = torch.randint(0, 256, (n_out, n_in // 2), generator=g, device=self.device, dtype=torch.uint8)
            sc = ((torch.rand(n_out, n_in // group_size, generator=g, device=self.device) * 0.5 + 0.75) * (0.02 * 3.46 / 7.5)).to(self.dtype)
            zp = torch.randint(7, 10, (n_out, n_in // group_size), generator=g, device=self.device, dtype=torch.uint8)
            return qw, sc, zp

        d, H, I = self.d, self.H, self.I
        for l in range(self.L):
            p = f"model.layers.{l}."
            parts = {}
            for name, (n_out, n_in) in (("self_attn.q_proj", (self.nh * d, H)), ("self_attn.k_proj", (self.nkv * d, H)), ("self_attn.v_proj", (self.nkv * d, H)),
                                        ("self_attn.o_proj", (H, self.nh * d)), ("mlp.gate_proj", (I, H)), ("mlp.up_proj", (I, H)), ("mlp.down_proj", (H, I))):
                t = make(n_out, n_in)
                packed[p + name] = t
                if not w4_only:
                    parts[name] = dequantize_w4(*t, group_size)
            if w4_only:
                continue
            self.wqkv[l].copy_(torch.cat([parts["self_attn.q_proj"], parts["self_attn.k_proj"], parts["self_attn.v_proj"]], 0))
            self.wo[l].copy_(parts["self_attn.o_proj"])
            gp, up = parts["mlp.gate_proj"], parts["mlp.up_proj"]
            self.wgu[l].copy_(torch.stack([gp.view(-1, 64, H), up.view(-1, 64, H)], 1).reshape(2 * I, H))
            self.wd[l].copy_(parts["mlp.down_proj"])
            del parts
        return self.attach_w4(packed, group_size, w4_only=w4_only)

    # ------------------------------------------------------------------------------------------ layers
    def _splits(self, T):
        c = self.ctx
        import os
        ov = os.environ.get("CTS_SPLITS")          # tuning override "qkv,o,gu,d" (decode-sized T only)
        if ov and T <= 32:
            a = [int(v) for v in ov.split(",")]
            return dict(qkv=a[0], o=a[1], gu=a[2], d=a[3])
        return dict(qkv=c.suggest_split(self.n_qkv, self.H, T), o=c.suggest_split(self.H, self.nh * self.d, T),
                    gu=c.suggest_split(self.I, self.H, T, True), d=c.suggest_split(self.H, self.I, T))

    def _ws_floats(self, T, sp):
        return max(sp["qkv"] * T * self.n_qkv if sp["qkv"] > 1 else 0, sp["o"] * T * self.H if sp["o"] > 1 else 0,
                   sp["gu"] * T * 2 * self.I if T <= 128 else 0, sp["d"] * T * self.H if sp["d"] > 1 else 0, 1)

    def _w4_splits(self, T):
        """Split-K factors of the four projections for a W4A16 decode step of T tokens."""
        w4, c = self.w4, self.ctx
        if w4["splits"] is not None:
            return w4["splits"]
        return dict(qkv=c.gemm_w4_mma_suggest_split(self.n_qkv, self.H, T), o=c.gemm_w4_mma_suggest_split(self.H, self.nh * self.d, T),
                    gu=c.gemm_w4_mma_suggest_split(2 * self.I, self.H, T), d=c.gemm_w4_mma_suggest_split(self.H, self.I, T))

    def _layers(self, st, T, attend):
        """Runs every decoder layer on st.h [T,H] in place; leaves RMSNorm_final(h) in st.xn."""
        c, sp, eps = self.ctx, st.splits, self.eps
        I, H = self.I, self.H
        c.reduce_residual_rmsnorm(None, 0, st.h, None, self.ln1[0], eps, st.xn, t=T)
        fused = self.use_fused_decode and T <= 32 and st.k_lin is None                            # decode states only
        # decode-sized steps: every weight-streaming GEMM names the weight its successor will stream, and prefetches the head of it
        # into L2 once its own last tile is requested (cts_gemm_args.next_*): HBM keeps streaming through the kernel boundaries
        nb = self.next_prefetch_bytes if (T <= 32 and st.k_lin is None) else 0
        # W4A16: decode-sized steps stream the 4-bit codes (every projection through the split-K partial path with the W4 split factors)
        w4 = self.w4 if (self.w4 is not None and T <= 32 and st.k_lin is None and not fused) else None
        if w4 is not None:
            sp = self._w4_splits(T)
        # 4-bit-only models: every other step (prefill of any length, decode batches of 33-128 rows) runs the projections through
        # cts_gemm_w4_prefill with exactly the epilogue and split factor the dense path below chooses -- the same numbers, bit for bit
        w4p = self.w4 if (self.w4 is not None and self.w4["only"] and w4 is None) else None

        def gemm(kind, l, x, w, out, **kw):
            """One projection: the dense GEMM on ``w``, or the 4-bit weight of (kind, l) with the same epilogue (4-bit-only models)."""
            if w4p is None:
                c.gemm(x, w, out, **kw)
                return
            qwf, szp, n_out = w4p[kind][l]
            kw = {k: v for k, v in kw.items() if not k.startswith("next_")}
            c.gemm_w4_prefill(x, qwf, szp, n_out, w4p["group_size"], out, **kw)

        def proj(kind, l, x, w, split, **kw):
            """fp32 split-K partials of one projection into st.ws: from the packed 4-bit weight when attached, else from the dense one."""
            if w4 is not None and w4["kernel"] == "mma":
                qwf, szp, n_out = w4[kind][l]
                c.gemm_w4_mma(x, qwf, szp, n_out, w4["group_size"], st.ws, split, t=T)
            elif w4 is not None:
                qw, sc, zp = w4[kind][l]
                c.gemm_w4(x, qw, sc, zp, w4["group_size"], st.ws, split, t=T)
            else:
                gemm(kind, l, x, w, st.ws, epilogue=EPI_PARTIAL_F32, split_k=split, t=T, **kw)

        def nxt(w, split):
            return dict(next_w=w, next_split=split, next_bytes=nb) if nb > 0 else {}
        for l in range(self.L):
            kc, vc = self.kv[l, 0], self.kv[l, 1]
            if fused:
                # 7 stages per layer: every projection reduces its K splits inside a cluster and applies its tail in the epilogue
                # (under tensor parallelism the row-parallel o_proj / down_proj keep the peer-memory all-reduce kernel, which sums
                # the local splits itself; the column-parallel QKV and gate_up projections are fused all the same)
                nw = self.ln1[l + 1] if l + 1 < self.L else self.final_norm
                # level 2 under tensor parallelism: the row-parallel projections carry their all-reduce INSIDE the GEMM kernel
                # (gemm_decode_fused peer tail; needs the low-latency regions, use_peer_ll) -- 5 launches per layer, none of them a collective
                tp_deep = self.tp_size > 1 and self.use_peer_ll and self.peer is not None and H % (128 * self.tp_size) == 0
                deep = self.use_fused_decode >= 2 and (self.tp_size == 1 or tp_deep)
                pr = [None, None]
                so, sd = min(sp["o"], 8), min(sp["d"], 8)
                if deep and self.tp_size > 1:
                    # a (tile, token) of the in-kernel all-reduce waits for the same tile's CTAs on the other ranks: keep every rank's
                    # whole grid resident (one CTA per SM suffices) instead of relying on the order CTAs are scheduled in
                    cap = max(1, 148 // max(1, H // 128))
                    so, sd = min(so, cap), min(sd, cap)
                    pr = [(self.peer.partials[w], self.peer.part_bytes, self.peer.state, self.tp_rank, self.tp_size, self.peer.max_batch) for w in (0, 1)]
                rope = dict(bias=self.bqkv[l], positions=st.positions, cos=self.cos, sin=self.sin, slot_map=st.slot_map, q_out=st.q, k_cache=kc,
                            v_cache=vc, q_norm=self.qn[l], k_norm=self.kn[l], eps=eps, nh=self.nh, nkv=self.nkv, head_dim=self.d,
                            page_size=self.page_size)
                if deep:
                    # 5 stages: QKV(norm in, RoPE out) -> attention -> o_proj(+residual, sum of squares out) -> gate_up(norm in, SwiGLU out)
                    # -> down(+residual, sum of squares out); layer 0 takes the xn of the plain RMSNorm above
                    if l == 0:
                        c.gemm_decode_fused(st.xn, self.wqkv[l], _cabi.FUSED_QKV_ROPE, min(sp["qkv"], 8), T, **rope)
                    else:
                        c.gemm_decode_fused(None, self.wqkv[l], _cabi.FUSED_QKV_ROPE, min(sp["qkv"], 8), T, norm_h=st.h, norm_w=self.ln1[l],
                                            ssq_in=st.ssq_b, norm_eps=eps, **rope)
                    attend(l)
                    c.gemm_decode_fused(st.ao, self.wo[l], _cabi.FUSED_RESIDUAL, so, T, h=st.h, ssq_out=st.ssq_a, peer=pr[0])
                    c.gemm_decode_fused(None, self.wgu[l], _cabi.FUSED_SWIGLU, min(sp["gu"], 8), T, act=st.act, norm_h=st.h, norm_w=self.ln2[l],
                                        ssq_in=st.ssq_a, norm_eps=eps)
                    c.gemm_decode_fused(st.act, self.wd[l], _cabi.FUSED_RESIDUAL, sd, T, h=st.h, ssq_out=st.ssq_b, peer=pr[1])
                    if l + 1 == self.L:
                        c.reduce_residual_rmsnorm(None, 0, st.h, None, self.final_norm, eps, st.xn, t=T)
                    continue
                c.gemm_decode_fused(st.xn, self.wqkv[l], _cabi.FUSED_QKV_ROPE, min(sp["qkv"], 8), T, **rope)
                attend(l)
                if self.tp_size > 1:
                    self._tp_row_parallel(st, T, st.ao, self.wo[l], self.ln2[l], 0, sp["o"])
                else:
                    c.gemm_decode_fused(st.ao, self.wo[l], _cabi.FUSED_RESIDUAL, min(sp["o"], 8), T, h=st.h)
                    c.reduce_residual_rmsnorm(None, 0, st.h, None, self.ln2[l], eps, st.xn, t=T)
                c.gemm_decode_fused(st.xn, self.wgu[l], _cabi.FUSED_SWIGLU, min(sp["gu"], 8), T, act=st.act)
                if self.tp_size > 1:
                    self._tp_row_parallel(st, T, st.act, self.wd[l], nw, 1, sp["d"])
                else:
                    c.gemm_decode_fused(st.act, self.wd[l], _cabi.FUSED_RESIDUAL, min(sp["d"], 8), T, h=st.h)
                    c.reduce_residual_rmsnorm(None, 0, st.h, None, nw, eps, st.xn, t=T)
                continue
            # ---- QKV projection + bias + RoPE + KV write
            if sp["qkv"] > 1 or w4 is not None:
                proj("qkv", l, st.xn, self.wqkv[l], sp["qkv"], **nxt(self.wo[l], sp["o"]))
                c.qkv_rope_cache(st.ws, True, sp["qkv"], self.bqkv[l], st.positions, self.cos, self.sin, st.slot_map, st.q, kc, vc,
                                 st.k_lin, st.v_lin, T, self.nh, self.nkv, self.d, self.page_size, self.qn[l], self.kn[l], eps)
            else:
                gemm("qkv", l, st.xn, self.wqkv[l], st.qkv, bias=self.bqkv[l], epilogue=EPI_NONE, t=T, **nxt(self.wo[l], sp["o"]))
                c.qkv_rope_cache(st.qkv, False, 1, None, st.positions, self.cos, self.sin, st.slot_map, st.q, kc, vc,
                                 st.k_lin, st.v_lin, T, self.nh, self.nkv, self.d, self.page_size, self.qn[l], self.kn[l], eps)
            attend(l)
            # ---- o_proj + residual + post-attention RMSNorm
            if self.tp_size > 1:
                self._tp_row_parallel(st, T, st.ao, self.wo[l], self.ln2[l], 0, sp["o"], nxt(self.wgu[l], sp["gu"]))
            elif sp["o"] > 1 or w4 is not None:
                proj("o", l, st.ao, self.wo[l], sp["o"], **nxt(self.wgu[l], sp["gu"]))
                c.reduce_residual_rmsnorm(st.ws, sp["o"], st.h, st.h, self.ln2[l], eps, st.xn, t=T)
            else:
                gemm("o", l, st.ao, self.wo[l], st.h, residual=st.h, epilogue=EPI_RESIDUAL, t=T, **nxt(self.wgu[l], sp["gu"]))
                c.reduce_residual_rmsnorm(None, 0, st.h, None, self.ln2[l], eps, st.xn, t=T)
            # ---- gate/up + SwiGLU
            if T > 128:
                gemm("gu", l, st.xn, self.wgu[l], st.act, epilogue=EPI_SWIGLU_IL, t=T)   # persistent, SwiGLU fused in the tile
            else:
                proj("gu", l, st.xn, self.wgu[l], sp["gu"], **nxt(self.wd[l], sp["d"]))
                c.reduce_swiglu(st.ws, sp["gu"], T, I, st.act, interleaved=True)
            # ---- down_proj + residual + next layer's input RMSNorm (or the final norm)
            nw = self.ln1[l + 1] if l + 1 < self.L else self.final_norm
            after = nxt(self.wqkv[l + 1], sp["qkv"]) if l + 1 < self.L else nxt(self.lm_head, 1)
            if self.tp_size > 1:
                self._tp_row_parallel(st, T, st.act, self.wd[l], nw, 1, sp["d"], after)
            elif sp["d"] > 1 or w4 is not None:
                proj("d", l, st.act, self.wd[l], sp["d"], **after)
                c.reduce_residual_rmsnorm(st.ws, sp["d"], st.h, st.h, nw, eps, st.xn, t=T)
            else:
                gemm("d", l, st.act, self.wd[l], st.h, residual=st.h, epilogue=EPI_RESIDUAL, t=T, **after)
                c.reduce_residual_rmsnorm(None, 0, st.h, None, nw, eps, st.xn, t=T)

    def _tp_row_parallel(self, st, T, x, w, norm_w, which, split, nxt=None):
        """Row-parallel projection under tensor parallelism: local split-K partials -> sum over splits and ranks ->
        residual + norm.  Decode-sized T: ONE kernel over NVLink peer memory (cts_peer_allreduce_residual_rmsnorm: each
        CTA reduces its token's local split-K partials into the symmetric buffer, signals, pulls the peers' rows; the
        buffers alternate between o_proj (0) and down_proj (1)).  Large prefill T: NCCL (bandwidth-bound) -- fp32 reduce-scatter over token
        shards + all-gather of the rounded result by default, see the branches below."""
        c = self.ctx
        big = split == 1 and not (self.peer is not None and T <= self.peer_tokens)
        if big and self.tp_prefill_exchange == "16bit":
            # Opt-in (CTS_TP_PREFILL_EXCHANGE=16bit): every rank rounds its projection to the model dtype and NCCL sums the ranks' outputs
            # in that dtype -- what vLLM's RowParallelLinear does (qwen2.py:100-116 / 168-174) -- half the bytes of the fp32 all-reduce:
            # e2e at TP4 1 850 -> 2 466 tok/s, and the prefill logits move from 1.2e-2 to 1.8e-2 of max from the single-GPU model
            # (profiles/r2_bench_tp4_prefill_exchange_*.json).  Not the default: the sum is re-rounded at every ring step.
            proj = st.tp_proj
            c.gemm(x, w, proj, epilogue=EPI_NONE, t=T)
            torch.distributed.all_reduce(proj[:T], group=self.comm)
            st.h[:T].add_(proj[:T])                               # residual add in the model dtype (one rounding, as the fused tail does)
            c.reduce_residual_rmsnorm(None, 0, st.h, st.h, norm_w, self.eps, st.xn, t=T)
            return
        if big and self.tp_prefill_exchange == "rs_ag" and self._nccl:
            # Default for prefill-sized T: the fp32 sum is kept (reduce-scatter of the fp32 partials over token shards, summed by NCCL in
            # fp32) and only the RESULT travels in the model dtype (all-gather of the rounded shards): three quarters of the bytes of the
            # fp32 all-reduce, the same numbers as the single-GPU path up to the order of the fp32 sum -- h = resid + dtype(sum).
            W = self.tp_size
            ct = -(-T // W)                                       # tokens per shard (the last shard is padded: st.ws / st.tp_proj hold W * ct rows)
            c.gemm(x, w, st.ws, epilogue=EPI_PARTIAL_F32, split_k=1, t=T, **(nxt or {}))
            part = st.ws.view(-1)[: W * ct * self.H]
            torch.distributed.reduce_scatter_tensor(st.tp_shard32, part, group=self.comm)
            st.tp_shard16.copy_(st.tp_shard32)                    # ONE rounding of the projection to the model dtype (cast = plumbing)
            torch.distributed.all_gather_into_tensor(st.tp_proj.view(-1)[: W * ct * self.H], st.tp_shard16, group=self.comm)
            st.h[:T].add_(st.tp_proj[:T])                         # residual add in the model dtype, as the fused tail does
            c.reduce_residual_rmsnorm(None, 0, st.h, st.h, norm_w, self.eps, st.xn, t=T)
            return
        c.gemm(x, w, st.ws, epilogue=EPI_PARTIAL_F32, split_k=split, t=T, **(nxt or {}))
        if self.peer is not None and T <= self.peer_tokens and self.use_peer_ll:
            c.peer_allreduce_ll(st.ws, split, self.peer.partials[which], self.peer.part_bytes, self.peer.state, self.tp_rank, self.tp_size,
                                self.peer.max_batch, st.h, st.h, norm_w, self.eps, st.xn, T)
            return
        if self.peer is not None and T <= self.peer_tokens:
            c.peer_allreduce_residual_rmsnorm(st.ws, split, self.peer.partials[which], self.peer.flags[which], self.peer.state,
                                              self.tp_rank, self.tp_size, self.peer.max_batch, st.h, st.h, norm_w, self.eps,
                                              st.xn, T)
            return
        part = st.ws[: T * self.H] if split == 1 else st.ws.view(-1)[: split * T * self.H].view(split, T * self.H).sum(0)
        torch.distributed.all_reduce(part, group=self.comm)
        c.reduce_residual_rmsnorm(part, 1, st.h, st.h, norm_w, self.eps, st.xn, t=T)

    def _alloc_step(self, T, decode):
        st = _Step()
        dev, dt = self.device, self.dtype
        st.splits = self._splits(T)
        st.h = torch.empty(T, self.H, device=dev, dtype=dt)
        st.xn = torch.empty(T, self.H, device=dev, dtype=dt)
        st.q = torch.empty(T, self.nh * self.d, device=dev, dtype=dt)
        st.ao = torch.empty(T, self.nh * self.d, device=dev, dtype=dt)
        st.act = torch.empty(T, self.I, device=dev, dtype=dt)
        st.tp_proj = st.tp_shard32 = st.tp_shard16 = None
        tp_pad = 0
        if self.tp_size > 1 and not decode:                     # row-parallel exchange of a prefill: token shards of ceil(T / W) rows
            ct = -(-T // self.tp_size)
            tp_pad = self.tp_size * ct
            st.tp_proj = torch.empty(tp_pad, self.H, device=dev, dtype=dt)
            st.tp_shard32 = torch.empty(ct * self.H, device=dev, dtype=torch.float32)
            st.tp_shard16 = torch.empty(ct * self.H, device=dev, dtype=dt)
        st.qkv = torch.empty(T, self.n_qkv, device=dev, dtype=dt) if st.splits["qkv"] == 1 else None
        ws_n = max(self._ws_floats(T, st.splits), T * self.H, tp_pad * self.H)
        if decode and self.w4 is not None and T <= 32:   # W4A16 decode: every projection through the partial path with the W4 split factors
            sp = self._w4_splits(T)
            ws_n = max(ws_n, sp["qkv"] * T * self.n_qkv, sp["o"] * T * self.H, sp["gu"] * T * 2 * self.I, sp["d"] * T * self.H)
        if decode and self.use_native_step:          # cts_decoder_step always takes the split-K partial path (also at factor 1)
            sp = st.splits
            ws_n = max(ws_n, sp["qkv"] * T * self.n_qkv, sp["o"] * T * self.H, sp["gu"] * T * 2 * self.I, sp["d"] * T * self.H)
        st.ws = torch.empty(ws_n, device=dev, dtype=torch.float32)                           # split-K partials [S, T, N]
        st.positions = torch.zeros(T, device=dev, dtype=torch.int32)
        st.slot_map = torch.zeros(T, device=dev, dtype=torch.int32)
        if decode:
            st.k_lin = st.v_lin = None
        else:
            st.k_lin = torch.empty(T, self.nkv * self.d, device=dev, dtype=dt)
            st.v_lin = torch.empty(T, self.nkv * self.d, device=dev, dtype=dt)
        return st

    # ------------------------------------------------------------------------------------------ prefill
    def _prepare_inputs(self, input_ids, attention_mask, timeseries, layout_kind="hf"):
        """Host side of A2/A3/A7: patch counts (one sync), merged layout, page allocation, H2D of the int maps."""
        cfg, dev = self.config, self.device
        ids_cpu = torch.as_tensor(input_ids).cpu().numpy()
        if ids_cpu.ndim == 1:
            ids_cpu = ids_cpu[None]
        am_cpu = None if attention_mask is None else torch.as_tensor(attention_mask).cpu().numpy()
        counts, cnt_h = None, np.zeros(0, dtype=np.int64)
        if timeseries is not None and timeseries.shape[0] > 0:
            if self.ts_encoder is None:
                raise ValueError("time series given but the checkpoint has no ts_encoder weights")
            if not isinstance(timeseries, torch.Tensor):
                raise ValueError(f"Incorrect type of ts input features. Got type: {type(timeseries)}")   # chatts_vllm.py:533-535
            counts = self.ts_encoder.patch_counts(timeseries)            # H2D (if needed) + count kernels, async
            host = torch.stack([counts[1], counts[2]]).cpu()             # the one host sync: (valid_len, patch_cnt)
            self._host_counts = (host[0], host[1])
            cnt_h = host[1].numpy().astype(np.int64)
        if layout_kind == "hf":
            import os as _os
            mode = _os.environ.get("CTS_TS_MERGE_MODE") or getattr(cfg, "ts_merge_mode", "insert")
            lay = layout.hf_layout(ids_cpu, am_cpu, cnt_h, cfg.ts_token_start_index, mode)
        else:
            lay = layout.vllm_layout(ids_cpu, int(cnt_h.sum()), cfg.ts_token_start_index)
        return ids_cpu, am_cpu, counts, lay

    def _prefill(self, lay, counts, timeseries, page_tables, all_logits=False):
        """Runs the prompt through the TS encoder + decoder, fills the paged KV cache, returns logits
        ([B,V] last position, or [T,V] for every merged position when all_logits)."""
        c, dev, dt = self.ctx, self.device, self.dtype
        T, B = lay.total, lay.cu_seqlens.shape[0] - 1
        lens = lay.lens
        if int(lens.max()) > self.n_pos:
            raise ValueError(f"prompt of {int(lens.max())} positions exceeds max_seq_len {self.n_pos}")
        st = self._alloc_step(T, decode=False)
        # slots of every prompt position in the paged cache
        b_of = np.repeat(np.arange(B), lens)
        pos = lay.positions.astype(np.int64)
        slot = page_tables[b_of, pos // self.page_size].astype(np.int64) * self.page_size + pos % self.page_size
        host = np.concatenate([lay.ids, lay.positions, slot.astype(np.int32), lay.cu_seqlens]).astype(np.int32)
        hbuf = torch.from_numpy(host).pin_memory()
        dbuf = hbuf.to(dev, non_blocking=True)
        ids_d, st.positions, st.slot_map, cu_d = dbuf[:T], dbuf[T:2 * T], dbuf[2 * T:3 * T], dbuf[3 * T:]
        c.embed_gather(self.embed, ids_d, st.h, t=T)
        if counts is not None and lay.row_map.shape[0] > 0:
            rmap = torch.from_numpy(lay.row_map).to(dev, non_blocking=True)
            self.ts_encoder.encode(timeseries, out=st.h, row_map=rmap, counts=counts, host_counts=self._host_counts)
        max_len = int(lens.max())
        scale = 1.0 / math.sqrt(self.d)

        def attend(l):
            c.attn_prefill(st.q, st.k_lin, st.v_lin, cu_d, B, max_len, self.nh, self.nkv, self.d, scale, st.ao)

        self._layers(st, T, attend)
        if all_logits:
            hn = st.xn
        else:
            last = torch.from_numpy((lay.cu_seqlens[1:] - 1).astype(np.int64)).to(dev)
            hn = st.xn.index_select(0, last).contiguous()        # row gather of B rows (plumbing)
        logits = torch.empty(hn.shape[0], self.V, device=dev, dtype=dt)
        c.gemm(hn, self.lm_head, logits, epilogue=EPI_NONE)
        return self._gather_vocab(logits)

    def _gather_vocab(self, logits):
        if self.tp_size == 1:
            return logits
        parts = [torch.empty_like(logits) for _ in range(self.tp_size)]
        torch.distributed.all_gather(parts, logits, group=self.comm)
        return torch.cat(parts, dim=-1)

    def forward(self, input_ids, attention_mask=None, timeseries=None, logits_to_keep=1, layout_kind="hf", **_):
        """HF-style forward.  layout_kind="hf": input_ids hold the un-expanded <ts><ts/> pairs, patch rows are inserted
        (HF surface); "vllm": one flat prompt whose <ts> copies are overwritten in order (chatts_vllm.py:405-415,569-573).
        logits_to_keep=1 -> [B,1,V] (next-token logits); 0 -> list of per-sample [T_b, V] tensors for every position."""
        _, _, counts, lay = self._prepare_inputs(input_ids, attention_mask, timeseries, layout_kind)
        B = lay.cu_seqlens.shape[0] - 1
        pts, held = self._alloc_pages(lay.lens, 0)
        try:
            logits = self._prefill(lay, counts, timeseries, pts, all_logits=(logits_to_keep == 0))
        finally:
            self.pool.release(held)
        if logits_to_keep == 0:
            cu = lay.cu_seqlens
            return CausalLMOutput([logits[cu[b]:cu[b + 1]] for b in range(B)])
        return CausalLMOutput(logits[:, None, :])

    __call__ = forward

    def _alloc_pages(self, lens, extra):
        B = len(lens)
        if B > self.max_batch:
            raise ValueError(f"batch {B} exceeds max_batch {self.max_batch}")
        pt = np.zeros((B, self.max_pages), dtype=np.int32)
        # all-or-nothing: every need is checked before the first page leaves the pool, so a failure can never strand pages
        # (ContinuousEngine._admit retries a RuntimeError; a leak there would shrink the pool for good)
        needs = []
        for b in range(B):
            n_tok = int(lens[b]) + extra
            if n_tok > self.n_pos:
                raise ValueError(f"sequence of {n_tok} tokens exceeds the {self.n_pos} positions of the rotary table "
                                 f"(min(max_position_embeddings, max_seq_len))")
            need = (n_tok + self.page_size - 1) // self.page_size
            if need > self.max_pages:
                raise ValueError(f"sequence of {n_tok} tokens exceeds max_seq_len {self.max_seq_len}")
            needs.append(need)
        if sum(needs) > len(self.pool.free):
            raise RuntimeError(f"KV cache exhausted: need {sum(needs)} pages, {len(self.pool.free)} free of {self.pool.num_pages}")
        held = []
        try:
            for b, need in enumerate(needs):
                pg = self.pool.alloc(need)
                held += pg
                pt[b, :need] = pg
        except BaseException:
            self.pool.release(held)
            raise
        return pt, held

    # ------------------------------------------------------------------------------------------ decode
    def _decode_state(self, B, max_new):
        key = B
        st = self._steps.get(key)
        if st is not None and st.out_tokens.shape[1] >= max_new:
            return st
        dev = self.device
        st = self._alloc_step(B, decode=True)
        st.B = B
        st.cur_ids = torch.zeros(B, device=dev, dtype=torch.int32)
        st.seq_lens = torch.zeros(B, device=dev, dtype=torch.int32)
        st.page_table = torch.zeros(B, self.max_pages, device=dev, dtype=torch.int32)
        st.out_tokens = torch.zeros(B, max(max_new, 256), device=dev, dtype=torch.int32)
        st.step_ptr = torch.zeros(2, device=dev, dtype=torch.int32)      # {step, arrival counter}
        st.logits = torch.empty(B, self.V, device=dev, dtype=self.dtype)
        # flash-decode split: fill the SMs with (split x kv head x batch) CTAs, at least 2 pages per split
        # (the kernel holds a 3-stage ring of 32 KB K+V tiles: TWO CTAs per SM; sizing for three gave 384 CTAs = two waves at TP2)
        per = max(1, (2 * 148) // max(1, B * self.nkv))
        max_tiles = max(1, (self.max_seq_len + 63) // 64)
        st.attn_splits = int(max(1, min(per, max_tiles, 32)))
        import os
        if os.environ.get("CTS_ATTN_SPLITS"):                      # tuning override
            st.attn_splits = int(os.environ["CTS_ATTN_SPLITS"])
        st.attn_ws = torch.zeros(self.ctx.attn_decode_workspace_floats(B, self.nh, self.d, st.attn_splits), device=dev,
                                 dtype=torch.float32)      # zero-filled once: holds the self-resetting split counters
        st.ssq = torch.zeros(B * 8, device=dev, dtype=torch.float32)
        tiles_h = (self.H + 127) // 128                             # per-tile sums of squares of h (fused decode level 2)
        st.ssq_a = torch.zeros(B, tiles_h, device=dev, dtype=torch.float32)
        st.ssq_b = torch.zeros(B, tiles_h, device=dev, dtype=torch.float32)
        st.chain_sync = torch.zeros(2, device=dev, dtype=torch.int32)       # grid-barrier counters of the chain kernel
        st.graph = st.graph_nosample = None
        self._steps[key] = st
        return st

    def _native_ok(self, B):
        return self.use_native_step and self.tp_size == 1 and B <= 128 and not self._chain_ok(B) and self.w4 is None

    def _chain_ok(self, B):
        return (self.w4 is None and self.use_chain and self.tp_size == 1 and B <= 32 and self.H % 64 == 0 and self.H // 64 <= 192 and self.I % 64 == 0)

    def _decode_layers_chain(self, st, attend):
        """Decode layers with the persistent chain kernel: per layer ONE attention launch + ONE chain launch
        (o_proj -> +resid/norm -> gate_up -> SwiGLU -> down -> +resid/norm -> next QKV -> RoPE/KV write)."""
        c, B, sp = self.ctx, st.B, st.splits
        common = dict(t=B, hidden=self.H, inter=self.I, nh=self.nh, nkv=self.nkv, head_dim=self.d,
                      splits=(sp["o"], sp["gu"], sp["d"], sp["qkv"]), h=st.h, xn=st.xn, act=st.act, ws=st.ws, ssq=st.ssq,
                      sync=st.chain_sync, eps=self.eps, dtype=self.dtype, positions=st.positions, cos=self.cos, sin=self.sin,
                      slot_map=st.slot_map, q_out=st.q, page_size=self.page_size)
        # head: RMSNorm(ln1[0]) -> QKV(0) -> RoPE / KV write(0)
        c.decode_chain(phases=(5, 8), norm5_has_partial=0, ln_next=self.ln1[0], wqkv=self.wqkv[0], bqkv=self.bqkv[0],
                       q_norm_w=self.qn[0], k_norm_w=self.kn[0], k_cache=self.kv[0, 0], v_cache=self.kv[0, 1], **common)
        for l in range(self.L):
            attend(l)
            last = l == self.L - 1
            nxt = {} if last else dict(wqkv=self.wqkv[l + 1], bqkv=self.bqkv[l + 1], q_norm_w=self.qn[l + 1], k_norm_w=self.kn[l + 1],
                                       k_cache=self.kv[l + 1, 0], v_cache=self.kv[l + 1, 1])
            c.decode_chain(phases=(0, 6 if last else 8), wo=self.wo[l], ao=st.ao, ln_post=self.ln2[l], wgu=self.wgu[l], wd=self.wd[l],
                           ln_next=self.final_norm if last else self.ln1[l + 1], **nxt, **common)

    def _decode_body(self, st, sample):
        c, B = self.ctx, st.B
        scale = 1.0 / math.sqrt(self.d)
        if self._native_ok(B):
            if not hasattr(self, "_layer_list"):
                self._layer_list = [dict(wqkv=self.wqkv[l], bqkv=self.bqkv[l], q_norm=self.qn[l], k_norm=self.kn[l], wo=self.wo[l],
                                         wgu=self.wgu[l], wd=self.wd[l], ln1=self.ln1[l], ln2=self.ln2[l], k_cache=self.kv[l, 0],
                                         v_cache=self.kv[l, 1]) for l in range(self.L)]
            sp = st.splits
            c.decoder_step(layers=self._layer_list, embed=self.embed, final_norm=self.final_norm, lm_head=self.lm_head, cos=self.cos,
                           sin=self.sin, hidden=self.H, inter=self.I, nh=self.nh, nkv=self.nkv, head_dim=self.d, eps=self.eps,
                           page_size=self.page_size, batch=B, splits=(sp["qkv"], sp["o"], sp["gu"], sp["d"]), attn_splits=st.attn_splits,
                           cur_ids=st.cur_ids, positions=st.positions, seq_lens=st.seq_lens, slot_map=st.slot_map, page_table=st.page_table,
                           out_tokens=st.out_tokens, step_ptr=st.step_ptr, h=st.h, xn=st.xn, q=st.q, ao=st.ao, act=st.act,
                           logits=st.logits, ws=st.ws, attn_ws=st.attn_ws, sample=sample)
            st.full_logits = st.logits
            return
        c.embed_gather(self.embed, st.cur_ids, st.h, t=B)

        def attend(l):
            c.attn_decode(st.q, self.kv[l, 0], self.kv[l, 1], st.page_table, st.seq_lens, B, self.nh, self.nkv, self.d,
                          self.page_size, scale, st.attn_splits, st.attn_ws, st.ao)

        if self._chain_ok(B):
            self._decode_layers_chain(st, attend)
        else:
            self._layers(st, B, attend)
        nb = self.next_prefetch_bytes if B <= 32 else 0
        c.gemm(st.xn, self.lm_head, st.logits, epilogue=EPI_NONE, t=B,
               **(dict(next_w=self.wqkv[0], next_split=st.splits["qkv"], next_bytes=nb) if nb > 0 else {}))
        if sample and self.peer is not None:
            # vocab-parallel greedy over peer memory: no collective call, graph-capturable
            c.peer_greedy_advance(st.logits, B, self.tp_rank, self.tp_size, self.peer.cand, self.peer.cand_flags, self.peer.cand_state,
                                  self.peer.max_batch, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map,
                                  st.page_table, self.page_size)
            return
        st.full_logits = self._gather_vocab(st.logits)           # identity on one GPU; all-gather of vocab shards under TP
        if sample:
            c.greedy_advance(st.full_logits, B, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map,
                             st.page_table, self.page_size)

    def _decode_step(self, st, sample=True):
        """One decode step for the whole batch; replays the captured CUDA graph when enabled."""
        if not self.use_cuda_graph or (self.tp_size > 1 and not (self.graph_with_tp and self.peer is not None and sample)):
            self._decode_body(st, sample)
            return
        attr = "graph" if sample else "graph_nosample"
        g = getattr(st, attr)
        if g is None:
            # warm-up on a side stream (sets kernel attributes, touches every buffer), then capture.  The warm-up
            # step really runs, so save/restore the device-side loop state around it.
            saved = [t.clone() for t in (st.cur_ids, st.positions, st.seq_lens, st.slot_map, st.step_ptr, st.out_tokens)]
            s = torch.cuda.Stream(device=self.device)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._decode_body(st, sample)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            for t, v in zip((st.cur_ids, st.positions, st.seq_lens, st.slot_map, st.step_ptr, st.out_tokens), saved):
                t.copy_(v)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._decode_body(st, sample)
            setattr(st, attr, g)
            # capture does not execute: state is intact
        g.replay()

    # ------------------------------------------------------------------------------------------ generate
    @torch.no_grad()
    def generate(self, input_ids=None, attention_mask=None, timeseries=None, max_new_tokens=None, max_length=None,
                 do_sample=None, temperature=None, top_p=None, top_k=None, streamer=None, eos_token_id=None, pad_token_id=None,
                 synced_gpus=False, sync_every=16, ignore_eos=False, seed=None, repetition_penalty=None, **_):
        """model.generate(**processor_out, max_new_tokens=...) -> LongTensor [B, S + new] whose first S columns are
        the ORIGINAL (un-expanded) input ids (README.md:102-103)."""
        cfg, dev = self.config, self.device
        gd = getattr(self, "generation_defaults", None)
        if gd:                                          # checkpoint defaults apply only where the caller said nothing
            if do_sample is None and gd.get("do_sample"):
                do_sample = True
                temperature = gd.get("temperature", 1.0) if temperature is None else temperature
                top_p = gd.get("top_p") if top_p is None else top_p
                top_k = gd.get("top_k") if top_k is None else top_k
            if eos_token_id is None and gd.get("eos_token_id") is not None:
                eos_token_id = gd["eos_token_id"]
            if pad_token_id is None and gd.get("pad_token_id") is not None:
                pad_token_id = gd["pad_token_id"]
            if max_new_tokens is None and max_length is None and gd.get("max_new_tokens"):
                max_new_tokens = gd["max_new_tokens"]
            if repetition_penalty is None and gd.get("repetition_penalty") is not None:
                repetition_penalty = gd["repetition_penalty"]
        ids_cpu, am_cpu, counts, lay = self._prepare_inputs(input_ids, attention_mask, timeseries)
        B, S = ids_cpu.shape
        if max_new_tokens is None:
            max_new_tokens = (max_length - S) if max_length is not None else 20
        max_new_tokens = int(max_new_tokens)
        if max_new_tokens <= 0:
            return torch.as_tensor(ids_cpu, dtype=torch.long)
        eos = cfg.eos_token_id if eos_token_id is None else eos_token_id
        eos_set = set(eos) if isinstance(eos, (list, tuple, set)) else {int(eos)}
        pad = cfg.pad_token_id if pad_token_id is None else pad_token_id
        if do_sample and temperature is None:
            temperature = 1.0                                   # HF GenerationConfig default when do_sample=True names no temperature
        greedy = not (do_sample and temperature > 0)
        if not greedy and seed is None:
            # an unseeded call draws a fresh seed (a fresh torch.Generator would start from the same default seed every time);
            # under tensor parallelism rank 0's seed is broadcast so every rank picks the same tokens
            seed = int.from_bytes(__import__("os").urandom(7), "little")
            if self.tp_size > 1:
                box = [seed]
                torch.distributed.broadcast_object_list(box, src=0, group=self.comm)
                seed = int(box[0])
        page_tables, held = self._alloc_pages(lay.lens, max_new_tokens)
        try:
            with span("cts.prefill"):
                logits = self._prefill(lay, counts, timeseries, page_tables)
            st = self._decode_state(B, max_new_tokens)
            lens32 = torch.from_numpy(lay.lens.astype(np.int32))
            st.page_table.copy_(torch.from_numpy(page_tables), non_blocking=True)
            st.positions.copy_(lens32 - 1, non_blocking=True)       # advanced to len by the first greedy_advance
            st.seq_lens.copy_(lens32, non_blocking=True)             # -> len + 1: cache length once the new token is written
            st.step_ptr.zero_()
            gen = torch.Generator(device=dev)
            if seed is not None:
                gen.manual_seed(int(seed))
            kseed = int(seed) if seed is not None else 0

            def sample(lg, step):
                if self.use_sample_kernel:
                    # temperature / top-k / top-p + multinomial + advance in one launch; the draw is a function of (seed, step, row)
                    self.ctx.sample_advance(lg, B, temperature, top_k or 0, 1.0 if top_p is None else top_p, kseed, st.out_tokens,
                                            st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map, st.page_table,
                                            self.page_size)
                else:
                    self._sample_advance(st, lg, step, temperature, top_p, gen, top_k)

            # repetition penalty (transformers RepetitionPenaltyLogitsProcessor, e.g. from generation_config.json): the ids that occur in
            # a row -- prompt (the un-expanded input_ids, as HF sees them) and generated -- live in a device bit mask; every step's
            # logits are rewritten by cts_rep_penalty_apply before the argmax / sampling kernel, the new token is marked after it
            rep = float(repetition_penalty) if repetition_penalty not in (None, 1, 1.0) else None
            seen = None
            if rep is not None:
                Vfull = self.config.vocab_size
                seen = torch.zeros(B, (Vfull + 31) // 32, dtype=torch.int32, device=dev)
                am = np.ones_like(ids_cpu) if am_cpu is None else am_cpu
                rr, cc = np.nonzero(am)
                self.ctx.rep_penalty_mark(torch.from_numpy(ids_cpu[rr, cc].astype(np.int32)).to(dev), torch.from_numpy(rr.astype(np.int32)).to(dev),
                                          seen, Vfull)
                self.ctx.rep_penalty_apply(logits, B, seen, rep)

            def advance(lg, step):
                if greedy:
                    self.ctx.greedy_advance(lg, B, st.out_tokens, st.step_ptr, st.cur_ids, st.positions, st.seq_lens, st.slot_map,
                                            st.page_table, self.page_size)
                else:
                    sample(lg, step)
                if seen is not None:
                    self.ctx.rep_penalty_mark(st.cur_ids, None, seen, self.config.vocab_size)

            advance(logits, 0)
            done = np.zeros(B, dtype=bool)
            out = np.full((B, max_new_tokens), pad, dtype=np.int64)
            emitted = 0
            produced = 1
            chunk = 1 if streamer is not None else max(1, int(sync_every))
            while True:
                # flush what has been produced since the last sync
                if produced - emitted >= chunk or produced >= max_new_tokens:
                    toks = st.out_tokens[:, emitted:produced].cpu().numpy()      # D2H (sync)
                    for j in range(toks.shape[1]):
                        col = toks[:, j]
                        out[~done, emitted + j] = col[~done]
                        if streamer is not None:
                            streamer.put(torch.as_tensor(col))
                        if not ignore_eos:
                            done |= np.isin(col, list(eos_set))
                    emitted = produced
                    if produced >= max_new_tokens or done.all():
                        break
                with span("cts.decode_step"):
                    if greedy and seen is None:
                        self._decode_step(st, sample=True)
                    else:
                        self._decode_step(st, sample=False)
                        if seen is not None:
                            self.ctx.rep_penalty_apply(st.full_logits, B, seen, rep)
                        advance(st.full_logits, produced)
                produced += 1
            if streamer is not None:
                streamer.end()
        finally:
            self.pool.release(held)
        is_eos = np.isin(out[:, :emitted], list(eos_set)) if not ignore_eos else np.zeros((B, emitted), dtype=bool)
        first = np.where(is_eos.any(axis=1), is_eos.argmax(axis=1) + 1, emitted)
        n_out = int(min(max(first.max(), 1), max_new_tokens))
        return torch.cat([torch.as_tensor(ids_cpu, dtype=torch.long), torch.as_tensor(out[:, :n_out])], dim=1)

    def _sample_advance(self, st, logits, step, temperature, top_p, gen, top_k=None):
        """Stochastic sampling (temperature / top-p, chatts/utils/inference_tsmllm_deepspeed.py:95-100).  Round 1: the
        distribution arithmetic is torch on the device logits (not graph-captured); greedy is the fused kernel."""
        lg = logits[: st.B].float() / float(temperature)
        if top_k is not None and 0 < top_k < lg.shape[-1]:
            kth = torch.topk(lg, int(top_k), dim=-1).values[:, -1:]
            lg = lg.masked_fill(lg < kth, float("-inf"))
        probs = torch.softmax(lg, dim=-1)
        if top_p is not None and top_p < 1.0:
            sp, si = torch.sort(probs, dim=-1, descending=True)
            keep = (torch.cumsum(sp, dim=-1) - sp) < top_p
            sp = sp * keep
            probs = torch.zeros_like(probs).scatter_(1, si, sp)
            probs = probs / probs.sum(dim=-1, keepdim=True)
        tok = torch.multinomial(probs, 1, generator=gen).reshape(-1).to(torch.int32)
        st.out_tokens[:, step] = tok
        st.cur_ids.copy_(tok)
        st.positions.add_(1)
        st.seq_lens.add_(1)
        pg = torch.div(st.positions, self.page_size, rounding_mode="floor").long().clamp_(max=self.max_pages - 1)
        st.slot_map.copy_((st.page_table.gather(1, pg[:, None]).reshape(-1) * self.page_size +
                           st.positions % self.page_size).to(torch.int32))
        st.step_ptr[0] += 1
