"""Weights: HF checkpoint names, a seeded synthetic factory (no checkpoint exists offline, SURVEY.md F1),
safetensors loading, and the tensor-parallel shard plan.

Names follow the checkpoint / the reference's mapper (chatts/vllm/chatts_vllm.py:454-470,612-625):
  model.embed_tokens.weight, model.layers.{i}.self_attn.{q,k,v}_proj.{weight,bias}, ...o_proj.weight,
  model.layers.{i}.mlp.{gate,up,down}_proj.weight, ...{input,post_attention}_layernorm.weight,
  model.norm.weight, lm_head.weight (absent when tied, :619-623),
  ts_encoder.mlp.{0,2,..}.{weight,bias}, ts_encoder.position_embedding.weight.
"""
import glob
import os

import torch


def ts_encoder_shapes(cfg):
    ts = cfg.ts
    shapes = {}
    in_size = cfg.ts_input_size()
    for li in range(int(ts["num_layers"])):
        shapes[f"ts_encoder.mlp.{2 * li}.weight"] = (ts["hidden_size"], in_size)
        shapes[f"ts_encoder.mlp.{2 * li}.bias"] = (ts["hidden_size"],)
        in_size = ts["hidden_size"]
    if ts.get("use_position_embedding", False):
        shapes["ts_encoder.position_embedding.weight"] = (ts["max_sequence_length"] + 1, ts.get("embedding_dim", 16))
    return shapes


def decoder_shapes(cfg, layers=None):
    H, I, d = cfg.hidden_size, cfg.intermediate_size, cfg.head_dim
    nh, nkv = cfg.num_attention_heads, cfg.num_key_value_heads
    shapes = {"model.embed_tokens.weight": (cfg.vocab_size, H), "model.norm.weight": (H,)}
    if not cfg.tie_word_embeddings:
        shapes["lm_head.weight"] = (cfg.vocab_size, H)
    for l in range(cfg.num_hidden_layers if layers is None else layers):
        p = f"model.layers.{l}."
        shapes[p + "self_attn.q_proj.weight"] = (nh * d, H)
        shapes[p + "self_attn.k_proj.weight"] = (nkv * d, H)
        shapes[p + "self_attn.v_proj.weight"] = (nkv * d, H)
        if getattr(cfg, "attention_bias", True):
            shapes[p + "self_attn.q_proj.bias"] = (nh * d,)
            shapes[p + "self_attn.k_proj.bias"] = (nkv * d,)
            shapes[p + "self_attn.v_proj.bias"] = (nkv * d,)
        if getattr(cfg, "qk_norm", False):
            shapes[p + "self_attn.q_norm.weight"] = (d,)
            shapes[p + "self_attn.k_norm.weight"] = (d,)
        shapes[p + "self_attn.o_proj.weight"] = (H, nh * d)
        shapes[p + "mlp.gate_proj.weight"] = (I, H)
        shapes[p + "mlp.up_proj.weight"] = (I, H)
        shapes[p + "mlp.down_proj.weight"] = (H, I)
        shapes[p + "input_layernorm.weight"] = (H,)
        shapes[p + "post_attention_layernorm.weight"] = (H,)
    return shapes


def all_shapes(cfg):
    s = decoder_shapes(cfg)
    s.update(ts_encoder_shapes(cfg))
    return s


def synthetic_state_dict(cfg, seed=1234, device="cpu", dtype=torch.bfloat16, std=0.02, names=None):
    """Seeded random weights at the config's shapes (SURVEY.md §8d): N(0, std^2) for linears / embeddings /
    biases, U(0.5, 1.5) for norm weights (ones would hide a missing multiply).  Generated in fp32 on `device`
    with a torch.Generator, then cast -- so a CPU call gives the oracle and the GPU model identical values."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = {}
    for name, shape in all_shapes(cfg).items():
        if names is not None and name not in names:
            # still advance the generator identically? No: names-filtered dicts are only used for benchmarks.
            continue
        if name.endswith(("layernorm.weight", "q_norm.weight", "k_norm.weight")) or name == "model.norm.weight":
            t = torch.rand(shape, generator=g, device=device, dtype=torch.float32) + 0.5
        else:
            t = torch.randn(shape, generator=g, device=device, dtype=torch.float32) * std
        out[name] = t.to(dtype)
    return out


def load_checkpoint(path, device="cpu", dtype=None):
    """Read an HF checkpoint directory (config.json + *.safetensors [+ index]) into a name->tensor dict."""
    try:
        from safetensors import safe_open
    except ImportError as e:  # pragma: no cover
        raise RuntimeError("safetensors is required to load a checkpoint") from e
    files = sorted(glob.glob(os.path.join(path, "*.safetensors")))
    if not files:
        raise FileNotFoundError(f"no *.safetensors under {path}")
    sd = {}
    for f in files:
        with safe_open(f, framework="pt", device=str(device)) as sf:
            for k in sf.keys():
                t = sf.get_tensor(k)
                sd[k] = t.to(dtype) if dtype is not None and t.is_floating_point() else t
    return sd


# --------------------------------------------------------------------------------------------------
# GPTQ-Int4 checkpoints (README.md:52,262-263 advertise ChatTS-{8B,14B}-GPTQ-Int4; SURVEY.md 8(f) N2).
# Load-time dequantisation to the model dtype: the quantised checkpoints then run on the same bf16/fp16 kernels (same speed
# and memory as the full-precision model -- a W4A16 decode GEMM is not built).  Packing per AutoGPTQ / optimum's published
# `QuantLinear` (UNVERIFIED offline against a real checkpoint -- none is available; the CPU test is a pack/unpack round trip):
#   qweight int32 [in/8, out]   : 8 consecutive INPUT indices per word, low nibble first
#   qzeros  int32 [groups, out/8]: 8 consecutive OUTPUT indices per word; checkpoint_format "gptq" stores zero - 1
#   scales  fp16  [groups, out];  g_idx int32 [in] (group of every input row; absent = i // group_size)
#   W[out, in] = scales[g, out] * (q[in, out] - zero[g, out])
# --------------------------------------------------------------------------------------------------
def _unpack_nibbles(t, axis):
    """int32 words -> 8 four-bit values each, expanded along ``axis``."""
    sh = torch.arange(0, 32, 4, dtype=torch.int32, device=t.device)
    if axis == 0:
        v = (t[:, None, :] >> sh[None, :, None]) & 0xF
        return v.reshape(t.shape[0] * 8, t.shape[1])
    v = (t[:, :, None] >> sh[None, None, :]) & 0xF
    return v.reshape(t.shape[0], t.shape[1] * 8)


def dequantize_gptq_linear(qweight, qzeros, scales, g_idx=None, group_size=128, zero_offset=1, dtype=torch.bfloat16, scale_dtype=None):
    """scale_dtype: round the fp16 scales to this dtype first -- what the W4A16 decode kernel multiplies with (csrc/gemm_w4.cu), so that
    the dequantised copy the prefill uses and the on-the-fly dequantisation of the decode step are the same numbers (fp16: no-op)."""
    q = _unpack_nibbles(qweight.to(torch.int32), 0)                       # [in, out]
    z = _unpack_nibbles(qzeros.to(torch.int32), 1)[:, : scales.shape[1]] + int(zero_offset)   # [groups, out]
    n_in = q.shape[0]
    g = (torch.arange(n_in, device=q.device) // int(group_size)) if g_idx is None else g_idx.to(torch.long)
    sc = scales if scale_dtype is None else scales.to(scale_dtype)
    w = sc.to(torch.float32)[g] * (q - z[g]).to(torch.float32)            # [in, out]
    return w.t().contiguous().to(dtype)


# nibble position of K element j (0..7) inside a 32-bit word of the B200 layout: ((w >> 4 i) & 0x000F000F) yields the pair
# (k_2i, k_2i+1) in the low / high half-word, i.e. one 16-bit-pair per shift -- the form the magic-number int4 -> bf16/fp16
# conversion wants (csrc/gemm_w4.cu)
W4_NIBBLE_OF_K = (0, 4, 1, 5, 2, 6, 3, 7)


def repack_gptq_w4(qweight, qzeros, scales, group_size=128, zero_offset=1, dtype=torch.bfloat16):
    """GPTQ tensors of one Linear -> the K-major layout the W4A16 decode GEMM streams:
         qw  uint8 [out, in/2]   row n = the 4-bit codes of W[n, :], 8 consecutive K per 32-bit word in W4_NIBBLE_OF_K order
         sc  dtype [out, groups] scale of (row, group), rounded to the model dtype
         zp  uint8 [out, groups] integer zero point incl. the checkpoint's offset (W = sc * (q - zp))
       act-order checkpoints (a non-monotonic g_idx) are not representable here: the caller keeps the dequantised weight for them."""
    q = _unpack_nibbles(qweight.to(torch.int32), 0).t().contiguous()      # [out, in]
    n_out, n_in = q.shape
    assert n_in % 8 == 0
    q8 = q.view(n_out, n_in // 8, 8).to(torch.int64)
    word = torch.zeros(n_out, n_in // 8, dtype=torch.int64, device=q.device)
    for j, nib in enumerate(W4_NIBBLE_OF_K):
        word |= q8[:, :, j] << (4 * nib)
    qw = torch.stack([(word >> (8 * b)) & 0xFF for b in range(4)], dim=-1).to(torch.uint8).reshape(n_out, n_in // 2).contiguous()
    z = (_unpack_nibbles(qzeros.to(torch.int32), 1)[:, :n_out] + int(zero_offset)).t().contiguous()   # [out, groups]
    return qw, scales.t().contiguous().to(dtype), z.to(torch.uint8)


def dequantize_w4(qw, sc, zp, group_size=128):
    """Host statement of the kernel's on-the-fly dequantisation (tests): [out, in] in sc's dtype."""
    n_out, half = qw.shape
    b = qw.view(n_out, half // 4, 4).to(torch.int64)
    word = b[:, :, 0] | (b[:, :, 1] << 8) | (b[:, :, 2] << 16) | (b[:, :, 3] << 24)
    q = torch.stack([(word >> (4 * nib)) & 0xF for nib in W4_NIBBLE_OF_K], dim=-1).reshape(n_out, half * 2)
    g = torch.arange(half * 2, device=qw.device) // int(group_size)
    w = sc.to(torch.float32)[:, g] * (q - zp.to(torch.int64)[:, g]).to(torch.float32)
    return w.to(sc.dtype)


def _w4_codes(qw):
    """[out, in] integer codes of the row layout repack_gptq_w4 writes."""
    n_out, half = qw.shape
    b = qw.view(n_out, half // 4, 4).to(torch.int64)
    word = b[:, :, 0] | (b[:, :, 1] << 8) | (b[:, :, 2] << 16) | (b[:, :, 3] << 24)
    return torch.stack([(word >> (4 * nib)) & 0xF for nib in W4_NIBBLE_OF_K], dim=-1).reshape(n_out, half * 2)


W4_MMA_TILE = 256          # features per chunk of the fragment-major layout (csrc/gemm_w4_mma.cu: kTileN)


def repack_w4_mma(qw, sc, zp, group_size=128):
    """Row layout (repack_gptq_w4: qw uint8 [out, in/2], sc [out, groups], zp uint8 [out, groups]) -> the fragment-major layout the
    register-operand W4A16 kernel streams (include/chatts_b200.h: cts_gemm_w4f_args):
         qwf uint8 [ceil(out/256) * in/64 * 8192]  chunk (tile, kb) = 16 m-tiles x 32 lanes x 4 words; word (m, lane = 4 g + t, ks) holds the codes of
                                                   rows {g, g+8} of m-tile m at k = 64 kb + 16 ks + {2t, 2t+1, 2t+8, 2t+9}: nibble i < 4 is the
                                                   LOWER k of fragment register a_i (a_0: row g, k 2t; a_1: row g+8, k 2t; a_2: row g, k 2t+8;
                                                   a_3: row g+8, k 2t+8), nibble i + 4 the upper one
         szp int32 [ceil(out/256), groups, 256]    scale bits | (magic + zp) << 16  (magic: bf16 0x4300 = 128.0, fp16 0x6400 = 1024.0)
       Features beyond `out` are zero (scale 0)."""
    q = _w4_codes(qw)                                              # [out, in]
    n_out, n_in = q.shape
    assert n_in % 64 == 0 and n_in % int(group_size) == 0
    tiles = -(-n_out // W4_MMA_TILE)
    pad = tiles * W4_MMA_TILE - n_out
    if pad:
        q = torch.cat([q, torch.zeros(pad, n_in, dtype=q.dtype, device=q.device)], 0)
    # feature n = 256 tile + 16 m + 8 hi_row + g ; k = 64 kb + 16 ks + 8 k_hi + 2 t + k_odd
    v = q.view(tiles, 16, 2, 8, n_in // 64, 4, 2, 4, 2)            # [tile, m, hi_row, g, kb, ks, k_hi, t, k_odd]
    v = v.permute(0, 4, 1, 3, 7, 5, 8, 6, 2).contiguous()          # [tile, kb, m, g, t, ks, k_odd, k_hi, hi_row]: nibble = 4 k_odd + 2 k_hi + hi_row
    v = v.view(tiles, n_in // 64, 16, 32, 4, 8)
    word = torch.zeros(v.shape[:-1], dtype=torch.int64, device=q.device)
    for nib in range(8):
        word |= v[..., nib] << (4 * nib)
    qwf = torch.stack([(word >> (8 * b)) & 0xFF for b in range(4)], dim=-1).to(torch.uint8).reshape(-1).contiguous()
    magic = 0x4300 if sc.dtype == torch.bfloat16 else 0x6400
    sbits = sc.contiguous().view(torch.int16).to(torch.int64) & 0xFFFF           # [out, groups]
    pair = sbits | ((zp.to(torch.int64) + magic) << 16)
    if pad:
        pair = torch.cat([pair, torch.zeros(pad, pair.shape[1], dtype=pair.dtype, device=pair.device)], 0)
    pair = pair.view(tiles, W4_MMA_TILE, -1).permute(0, 2, 1).contiguous()      # [tile, group, 256]
    pair = torch.where(pair >= (1 << 31), pair - (1 << 32), pair).to(torch.int32)
    return qwf, pair


def dequantize_gptq(sd, quant_cfg=None, dtype=torch.bfloat16, scale_dtype=None):
    """Replace every ``<name>.{qweight,qzeros,scales[,g_idx]}`` group of a GPTQ checkpoint by ``<name>.weight``."""
    quant_cfg = quant_cfg or {}
    bits = int(quant_cfg.get("bits", 4))
    if bits != 4:
        raise ValueError(f"GPTQ checkpoints with {bits}-bit weights are not supported (4-bit only)")
    gs = int(quant_cfg.get("group_size", 128))
    zo = 0 if str(quant_cfg.get("checkpoint_format", "gptq")) == "gptq_v2" else 1
    out = {}
    for k, t in sd.items():
        if k.endswith(".qweight"):
            base = k[: -len(".qweight")]
            n_in = t.shape[0] * 8
            group = gs if gs > 0 else n_in                              # group_size -1: one group per column
            out[base + ".weight"] = dequantize_gptq_linear(t, sd[base + ".qzeros"], sd[base + ".scales"], sd.get(base + ".g_idx"),
                                                            group, zo, dtype, scale_dtype)
        elif k.endswith((".qzeros", ".scales", ".g_idx")) and (k.rsplit(".", 1)[0] + ".qweight") in sd:
            continue
        else:
            out[k] = t
    return out


def gptq_w4_pack(sd, quant_cfg=None, dtype=torch.bfloat16):
    """({linear name: (qw, scales, zeros)} in the W4A16 kernel's layout, group size) for a GPTQ checkpoint's decoder projections, or
    (None, 0) when the checkpoint cannot use the kernel: not 4-bit, an act-order g_idx, a group size that is not a multiple of 64, or
    linears that do not share one group size (group_size -1 = one group per input column: q/k/v/gate/up and o/down differ in n_in)."""
    quant_cfg = quant_cfg or {}
    if int(quant_cfg.get("bits", 4)) != 4:
        return None, 0
    gs = int(quant_cfg.get("group_size", 128))
    zo = 0 if str(quant_cfg.get("checkpoint_format", "gptq")) == "gptq_v2" else 1
    out, groups = {}, set()
    for k, t in sd.items():
        if not k.endswith(".qweight") or ".layers." not in k:
            continue
        base = k[: -len(".qweight")]
        n_in = t.shape[0] * 8
        group = gs if gs > 0 else n_in
        if group % 64 != 0 or n_in % group != 0:
            return None, 0
        gi = sd.get(base + ".g_idx")
        if gi is not None and not torch.equal(gi.to(torch.int64).cpu(), torch.arange(n_in) // group):
            return None, 0                                                # act-order: rows of one group are scattered over K
        out[base] = repack_gptq_w4(t, sd[base + ".qzeros"], sd[base + ".scales"], group, zo, dtype)
        groups.add(group)
    return (out, groups.pop()) if out and len(groups) == 1 else (None, 0)


def pack_gptq_linear(w, group_size=128, zero_offset=1):
    """Inverse of dequantize_gptq_linear for tests: asymmetric 4-bit round-to-nearest per (group, out) -> packed tensors."""
    wt = w.to(torch.float32).t().contiguous()                             # [in, out]
    n_in, n_out = wt.shape
    G = n_in // group_size
    wg = wt.view(G, group_size, n_out)
    lo, hi = wg.min(1).values, wg.max(1).values
    scale = ((hi - lo) / 15.0).clamp_min(1e-8)
    zero = torch.round(-lo / scale).clamp(0, 15)
    q = torch.clamp(torch.round(wg / scale[:, None]) + zero[:, None], 0, 15).to(torch.int32).view(n_in, n_out)
    sh = torch.arange(0, 32, 4, dtype=torch.int64)
    qweight = ((q.view(n_in // 8, 8, n_out).to(torch.int64) << sh[None, :, None]).sum(1) & 0xFFFFFFFF)
    zs = (zero.to(torch.int64) - zero_offset) & 0xF
    qzeros = ((zs.view(G, n_out // 8, 8) << sh[None, None, :]).sum(2) & 0xFFFFFFFF)
    to_i32 = lambda x: torch.where(x >= 2 ** 31, x - 2 ** 32, x).to(torch.int32)
    return to_i32(qweight), to_i32(qzeros), scale.to(torch.float16), (torch.arange(n_in) // group_size).to(torch.int32)


# --------------------------------------------------------------------------------------------------
# tensor parallel shard plan (Megatron style; SURVEY.md §8e): column split of QKV / gate / up / lm_head,
# row split of o_proj / down_proj, kv heads divided across ranks (nkv % tp == 0), everything else replicated.
# --------------------------------------------------------------------------------------------------
def shard_range(total, rank, size):
    assert total % size == 0, f"{total} not divisible by tensor-parallel size {size}"
    per = total // size
    return rank * per, (rank + 1) * per


def shard_tensor(name, t, cfg, rank, size):
    if size == 1:
        return t
    d = cfg.head_dim
    if name.endswith(("q_proj.weight", "q_proj.bias")):
        a, b = shard_range(cfg.num_attention_heads, rank, size)
        return t[a * d:b * d]
    if name.endswith(("k_proj.weight", "k_proj.bias", "v_proj.weight", "v_proj.bias")):
        a, b = shard_range(cfg.num_key_value_heads, rank, size)
        return t[a * d:b * d]
    if name.endswith("o_proj.weight"):
        a, b = shard_range(cfg.num_attention_heads, rank, size)
        return t[:, a * d:b * d]
    if name.endswith(("gate_proj.weight", "up_proj.weight")):
        a, b = shard_range(cfg.intermediate_size, rank, size)
        return t[a:b]
    if name.endswith("down_proj.weight"):
        a, b = shard_range(cfg.intermediate_size, rank, size)
        return t[:, a:b]
    if name == "lm_head.weight":
        a, b = shard_range(cfg.vocab_size, rank, size)
        return t[a:b]
    return t
