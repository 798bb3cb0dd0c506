"""Host logic of the LoRA fine-tune step (row A9) on CPU: chatts_b200.train.LoraTrainer driven through the torch test
double of the C-ABI, checked against oracle/lora.py (autograd over the decoder oracle): loss, every adapter gradient,
the AdamW update, gradient accumulation over micro-batches, label handling at the ``<ts>`` patch rows, the packed fused
operands, the peft adapter file round trip into merge_lora, and the record encoder."""
import json
import os

import numpy as np
import pytest
import torch

from chatts_b200 import ChatTSConfig, ChatTSProcessor, SimpleTokenizer
from chatts_b200.weights import synthetic_state_dict
from oracle import lora as ol
from oracle import merge as om
from oracle import ts_encoder as ote

DT = torch.bfloat16


def _series():
    x = np.arange(256)
    a = np.sin(x / 10) * 5.0
    a[100:] -= 10.0
    return a, (x * 0.05)[:100], np.cos(x / 7)[:48]


RECORDS = [
    {"input": "A <ts><ts/> and B <ts><ts/> ? ", "output": "first falls, second rises", "timeseries": [_series()[0], _series()[1]]},
    {"input": "Only text here, a longer prompt so that the other sample is left-padded: ", "output": "nothing to see", "timeseries": []},
    {"input": "C <ts><ts/>: ", "output": "a short wave", "timeseries": [_series()[2]]},
]


def _build(cabi_double, qwen3, **kw):
    from chatts_b200.model import ChatTSForCausalLM

    cfg = ChatTSConfig.tiny()
    if qwen3:
        cfg.qk_norm, cfg.attention_bias = True, False
    sd = synthetic_state_dict(cfg, seed=1234, device="cpu", dtype=DT, std=0.05)
    model = ChatTSForCausalLM(cfg, sd, device="cpu", dtype=DT, max_batch=8, max_seq_len=512, page_size=16, use_cuda_graph=False)
    proc = ChatTSProcessor(SimpleTokenizer(cfg.ts_token_start_index, cfg.pad_token_id, cfg.eos_token_id), cfg)
    return cfg, sd, model, proc


def _oracle_inputs(cfg, sd, batch):
    """Merged embeddings + merged labels per sample, by the oracle's own merge (oracle/merge.py)."""
    ts_w = {k[len("ts_encoder."):]: v for k, v in sd.items() if k.startswith("ts_encoder.")}
    if batch["timeseries"].shape[0]:
        feats, pc = ote.forward(batch["timeseries"].to(DT), cfg.ts, ts_w)
        pc = pc.tolist()
    else:
        feats, pc = torch.zeros(0, cfg.hidden_size, dtype=DT), []
    embeds = om.hf_merge(batch["input_ids"], batch["attention_mask"], sd["model.embed_tokens.weight"], feats, pc, cfg.ts_token_start_index)
    labels, k = [], 0
    for b in range(batch["input_ids"].shape[0]):
        out = []
        for col in range(batch["input_ids"].shape[1]):
            if not batch["attention_mask"][b, col]:
                continue
            out.append(int(batch["labels"][b, col]))
            if int(batch["input_ids"][b, col]) == cfg.ts_token_start_index:
                out += [-100] * int(pc[k])                     # patch rows follow <ts>; they are never learnt
                k += 1
        labels.append(torch.tensor(out, dtype=torch.long))
        assert labels[-1].shape[0] == embeds[b].shape[0]
    return embeds, labels


def _rel(a, b):
    return float((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-12))


@pytest.mark.parametrize("qwen3", [False, True])
def test_loss_and_gradients_match_oracle(cabi_double, qwen3):
    from chatts_b200.train import LoraTrainer, encode_records

    cfg, sd, model, proc = _build(cabi_double, qwen3)
    r, alpha = 8, 16
    tr = LoraTrainer(model, r=r, lora_alpha=alpha, seed=3, init_b_std=0.05, max_grad_norm=0.0)
    ad = ol.init_adapters(cfg.to_dict(), r, seed=3, b_std=0.05)
    for n, t in tr.adapters().items():                            # same generator order as the oracle's init
        assert torch.equal(t, ad[n]), n
    batch = encode_records(proc, RECORDS, eos_token_id=cfg.eos_token_id)
    assert LoraTrainer.count_labels(batch) == sum(len(proc.tokenizer.encode(r_["output"])) + 1 for r_ in RECORDS)
    tr.zero_grad()
    bt = tr.forward_backward(**batch)
    embeds, labels = _oracle_inputs(cfg, sd, batch)
    w = {k: v for k, v in sd.items() if not k.startswith("ts_encoder.")}
    loss, g = ol.grads(embeds, labels, w, ad, alpha / r, cfg.to_dict())
    assert bt.n_counted == LoraTrainer.count_labels(batch)
    assert abs(float(tr.loss_out[0]) - loss) < 2e-2 * abs(loss), (float(tr.loss_out[0]), loss)
    got = tr.grads()
    worst = {}
    for n, ref in g.items():
        assert ref.abs().max() > 0, n
        worst[n] = _rel(got[n], ref)
    bad = {n: e for n, e in worst.items() if e > 6e-2}           # two bf16 evaluations of a 2-layer forward + backward
    assert not bad, bad
    # cosine over the whole arena: direction of the step
    flat_ref = torch.cat([g[n].reshape(-1) for n in tr.index])
    cos = float(torch.nn.functional.cosine_similarity(tr.g, flat_ref, dim=0))
    assert cos > 0.999, cos


def test_optimizer_step_clip_and_accumulation(cabi_double):
    from chatts_b200.train import LoraTrainer, encode_records

    cfg, sd, model, proc = _build(cabi_double, True)
    kw = dict(r=8, lora_alpha=16, seed=5, init_b_std=0.05, lr=1e-2, betas=(0.9, 0.95), weight_decay=0.1)
    tr = LoraTrainer(model, max_grad_norm=0.05, **kw)
    full = encode_records(proc, RECORDS, eos_token_id=cfg.eos_token_id)
    p0 = tr.p.clone()
    loss_full = float(tr.train_step(full)[0])
    g_full, norm = tr.g.clone(), float(tr.norm_out[0])
    assert abs(norm - float(g_full.norm())) < 1e-4 * norm and norm > 0.05         # so the clip is active
    coef = 0.05 / (norm + 1e-6)
    pe, me, ve = ol.adamw_update(p0, g_full * coef, torch.zeros_like(p0), torch.zeros_like(p0), 1, lr=1e-2, betas=(0.9, 0.95),
                                 eps=1e-8, weight_decay=0.1)
    assert torch.allclose(tr.p, pe, atol=1e-6, rtol=1e-5) and torch.allclose(tr.m, me, atol=1e-7) and torch.allclose(tr.v, ve, atol=1e-9)
    # packed operands follow the master copy: B_f block of k_proj in layer 1 = bf16(alpha/r * B), transposed copy consistent
    g1 = tr.groups[1]["qkv"]
    mk = next(mm for mm in g1.members if mm.proj == "k_proj")
    bk = tr.param("model.layers.1.self_attn.k_proj.lora_B.weight")
    blk = g1.B[mk.n0: mk.n0 + mk.fout, mk.j0: mk.j0 + tr.r]
    assert torch.equal(blk, (bk * tr.scaling).to(DT)) and torch.equal(g1.Bt[mk.j0: mk.j0 + tr.r, mk.n0: mk.n0 + mk.fout], blk.T)
    assert float(g1.B[: mk.n0, mk.j0: mk.j0 + tr.r].abs().max()) == 0           # off-diagonal blocks stay zero
    ag = tr.param("model.layers.0.mlp.up_proj.lora_A.weight")
    gu = tr.groups[0]["gu"]
    mu = next(mm for mm in gu.members if mm.proj == "up_proj")
    assert torch.equal(gu.A[mu.j0: mu.j0 + tr.r], ag.to(DT)) and torch.equal(gu.At[:, mu.j0: mu.j0 + tr.r], ag.to(DT).T)
    bu = tr.param("model.layers.0.mlp.up_proj.lora_B.weight")
    il = gu.B.view(-1, 2, 64, gu.R)[:, 1].reshape(-1, gu.R)                      # "up" rows of the interleaved layout
    assert torch.equal(il[:, mu.j0: mu.j0 + tr.r], (bu * tr.scaling).to(DT))
    # micro-batches: same step from [records 0,1] + [record 2] as from the full batch (token-mean over the union)
    tr2 = LoraTrainer(model, max_grad_norm=0.05, **kw)
    mb = [encode_records(proc, RECORDS[:2], eos_token_id=cfg.eos_token_id), encode_records(proc, RECORDS[2:], eos_token_id=cfg.eos_token_id)]
    loss_mb = float(tr2.train_step(mb)[0])
    assert abs(loss_mb - loss_full) < 2e-3 * abs(loss_full)
    assert _rel(tr2.g, g_full) < 2e-2
    norm2 = float(tr2.norm_out[0])
    pe2, me2, ve2 = ol.adamw_update(p0, tr2.g * (0.05 / (norm2 + 1e-6)), torch.zeros_like(p0), torch.zeros_like(p0), 1, lr=1e-2,
                                    betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1)
    assert tr2.step_count == 1 and torch.allclose(tr2.p, pe2, atol=1e-6, rtol=1e-5)
    assert torch.allclose(tr2.m, me2, atol=1e-7) and torch.allclose(tr2.v, ve2, atol=1e-9)
    # the first Adam step moves every element by ~lr * sign(g): where |g| lies within the two gradients' disagreement (bf16 forwards of
    # differently padded batches, whose reduction order follows the host's thread count) the sign may differ, so those elements may
    # step up to 2 lr apart; everywhere else the two steps agree
    resolved = g_full.abs() > (tr2.g - g_full).abs().max()
    assert float(resolved.float().mean()) > 0.9
    assert torch.allclose(tr2.p[resolved], tr.p[resolved], atol=2e-4) and float((tr2.p - tr.p).abs().max()) < 2e-2


def test_training_reduces_the_loss_and_adapter_roundtrip(cabi_double, tmp_path):
    from chatts_b200.train import LoraTrainer, encode_records, load_jsonl, shard_records

    cfg, sd, model, proc = _build(cabi_double, False)
    path = tmp_path / "train.jsonl"
    with open(path, "w") as f:
        for r_ in RECORDS:
            f.write(json.dumps({**r_, "timeseries": [np.asarray(t).tolist() for t in r_["timeseries"]]}) + "\n")
    recs = load_jsonl(str(path))
    assert len(recs) == 3 and shard_records(recs, 1, 2) == [recs[1]]
    batch = encode_records(proc, recs, eos_token_id=cfg.eos_token_id)
    tr = LoraTrainer(model, r=8, lora_alpha=16, seed=0, lr=5e-3, max_grad_norm=1.0)       # peft init: B = 0
    l0 = float(tr.eval_loss(batch)[0])
    losses = [float(tr.train_step(batch)[0]) for _ in range(4)]
    assert abs(losses[0] - l0) < 1e-3 * l0                                               # B = 0: the adapters start as a no-op
    assert losses[-1] < losses[0] - 0.05, losses
    # first step with B = 0 moves only B (dA = 0 exactly)
    out = tmp_path / "adapter"
    tr.save_adapter(str(out))
    assert json.load(open(out / "adapter_config.json"))["r"] == 8
    # merged inference == adapter forward: logits of the merged model vs the training forward's loss on the same batch
    lt = float(tr.eval_loss(batch)[0])
    n = model.merge_lora(str(out))
    assert n == cfg.num_hidden_layers * 7
    tr0 = LoraTrainer(model, r=8, lora_alpha=16, seed=0)                                  # fresh B = 0 adapters on the MERGED weights
    lm = float(tr0.eval_loss(batch)[0])
    assert abs(lm - lt) < 3e-2 * lt, (lm, lt)


def test_label_rows_skip_patch_rows_and_sample_boundaries(cabi_double):
    from chatts_b200.train import LoraTrainer, encode_records

    cfg, sd, model, proc = _build(cabi_double, False)
    tr = LoraTrainer(model, r=8, seed=0)
    batch = encode_records(proc, RECORDS, eos_token_id=cfg.eos_token_id)
    bt = tr._prepare(batch["input_ids"], batch["attention_mask"], batch["timeseries"], batch["labels"])
    lay = bt.lay
    # every selected row is a text position or the LAST patch row before a text token; its target is that sample's next label
    assert bt.n_counted == LoraTrainer.count_labels(batch)
    ends = set((lay.cu_seqlens[1:] - 1).tolist())
    assert not ends & set(bt.sel.tolist())                                        # the last position of a sample predicts nothing
    for row, tgt in zip(bt.sel.tolist(), bt.targets.tolist()):
        assert lay.src_col[row + 1] >= 0 and tgt >= 0
    with pytest.raises(ValueError):
        tr.forward_backward(batch["input_ids"], batch["attention_mask"], batch["timeseries"], batch["labels"][:, :-1])


def test_fit_schedule_accumulation_and_resume(cabi_double, tmp_path):
    """fit(): seeded epochs over the shard, micro-batch accumulation, LR schedule identical to transformers', checkpoint +
    resume reproduces the uninterrupted run bit for bit."""
    from transformers.optimization import get_cosine_schedule_with_warmup, get_linear_schedule_with_warmup
    from chatts_b200.train import LoraTrainer, lr_factor

    for name, mk in (("cosine", get_cosine_schedule_with_warmup), ("linear", get_linear_schedule_with_warmup)):
        opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=1.0)
        sch = mk(opt, num_warmup_steps=3, num_training_steps=20)
        for step in range(20):
            assert abs(sch.get_last_lr()[0] - lr_factor(step, 20, 3, name)) < 1e-9, (name, step)
            opt.step(); sch.step()
    cfg, sd, model, proc = _build(cabi_double, False)
    recs = RECORDS * 2                                              # 6 records: 3 steps of 2 samples per epoch
    kw = dict(r=8, lora_alpha=16, seed=1, init_b_std=0.02, lr=5e-3, max_grad_norm=1.0)
    seen = []
    tr = LoraTrainer(model, **kw)
    full = tr.fit(proc, recs, epochs=2, samples_per_step=2, micro_batch=1, warmup_steps=2, eos_token_id=cfg.eos_token_id,
                  on_step=lambda s, l, t: seen.append((s, t.lr)))
    assert len(full) == 6 and tr.step_count == 6 and [s for s, _ in seen] == list(range(6))
    assert seen[0][1] == 0.0 and abs(seen[2][1] - 5e-3) < 1e-12 and seen[5][1] < seen[3][1] and tr.lr == 5e-3
    # interrupted after 4 steps, resumed from the checkpoint: same parameters as the uninterrupted run
    ck = str(tmp_path / "ck" / "trainer.pt")
    a = LoraTrainer(model, **kw)

    class Stop(Exception):
        pass

    def bail(s, l, t):
        if s == 3:
            t.save_checkpoint(ck)
            raise Stop

    with pytest.raises(Stop):
        a.fit(proc, recs, epochs=2, samples_per_step=2, micro_batch=1, warmup_steps=2, eos_token_id=cfg.eos_token_id, on_step=bail)
    b = LoraTrainer(model, **kw)
    rest = b.fit(proc, recs, epochs=2, samples_per_step=2, micro_batch=1, warmup_steps=2, eos_token_id=cfg.eos_token_id, checkpoint=ck)
    assert len(rest) == 2 and b.step_count == 6
    assert torch.equal(b.p, tr.p) and torch.equal(b.m, tr.m) and rest == full[4:]
    with pytest.raises(ValueError):
        LoraTrainer(model, r=4, seed=1).load_checkpoint(ck)


def test_gradient_is_the_directional_derivative(cabi_double):
    """No oracle involved: along D = g/|g|, (L(p + eD) - L(p - eD)) / 2e must equal |g| (the whole backward is the derivative
    of the loss the forward computes).  The same property is the GPU test at the ChatTS-8B layer shape."""
    from chatts_b200.train import LoraTrainer, encode_records

    cfg, sd, model, proc = _build(cabi_double, True)
    tr = LoraTrainer(model, r=8, lora_alpha=16, seed=2, init_b_std=0.02, max_grad_norm=0.0)
    batch = encode_records(proc, RECORDS, eos_token_id=cfg.eos_token_id)
    tr.zero_grad()
    tr.forward_backward(**batch)
    g, p0 = tr.g.clone(), tr.p.clone()
    D = g / g.norm()
    slope = float(g.norm())
    eps = 0.03 / slope
    vals = []
    for sgn in (1.0, -1.0):
        tr.p.copy_(p0 + sgn * eps * D)
        tr.pack()
        vals.append(float(tr.eval_loss(batch)[0]))
    fd = (vals[0] - vals[1]) / (2 * eps)
    assert abs(fd - slope) < 0.05 * slope, (fd, slope)


def test_label_rows_against_brute_force_on_random_batches(cabi_double):
    """_prepare (vectorised index arithmetic) vs a position-by-position statement of ForCausalLMLoss's shift on the merged
    sequence, over random batches: random texts with 0..3 series of ragged lengths, random output lengths, left padding."""
    from chatts_b200.train import LoraTrainer, encode_records

    cfg, sd, model, proc = _build(cabi_double, False)
    tr = LoraTrainer(model, r=8, seed=0)
    rng = np.random.default_rng(7)
    for trial in range(12):
        recs = []
        for _ in range(int(rng.integers(1, 5))):
            n_ts = int(rng.integers(0, 4))
            text = "".join(f"w{int(rng.integers(0, 99))} <ts><ts/> " for _ in range(n_ts)) + "q" * int(rng.integers(1, 30))
            series = [np.sin(np.arange(int(rng.integers(5, 200))) / 3.0) * float(rng.uniform(0.5, 9)) for _ in range(n_ts)]
            recs.append({"input": text, "output": "a" * int(rng.integers(1, 20)), "timeseries": series})
        batch = encode_records(proc, recs, eos_token_id=cfg.eos_token_id)
        bt = tr._prepare(batch["input_ids"], batch["attention_mask"], batch["timeseries"], batch["labels"])
        _, labels = _oracle_inputs(cfg, sd, batch)
        sel, tgt, base = [], [], 0
        for y in labels:                                   # position i of a sample predicts label i + 1 of the same sample
            for i in range(len(y) - 1):
                if int(y[i + 1]) != -100:
                    sel.append(base + i)
                    tgt.append(int(y[i + 1]))
            base += len(y)
        assert bt.sel.tolist() == sel and bt.targets.tolist() == tgt, trial
        assert bt.T == base and bt.n_counted == LoraTrainer.count_labels(batch) == len(sel)
