"""LoRA fine-tune step of the ChatTS decoder on B200 (SURVEY.md 8(a) row A9, BASELINE config 5: ChatTS-8B, forward +
backward on ``{input, output, timeseries}`` records, data parallel).

What the reference gives for this row: nothing executable -- training lives in the external ChatTS-Training project
(README.md:216-218); the repo only LOADS a peft adapter (demo/demo_lora.ipynb cells 3-4) and shows the record shape
(chatts/align/uts_template_qa.py:127-131).  So this module implements the published pieces that recipe is made of and is
checked against ``oracle/lora.py`` (torch.autograd over the decoder oracle, itself pinned against transformers):

  * peft ``lora.Linear``: y = W x + (alpha / r) B A x on q/k/v/o/gate/up/down_proj, base weights frozen;
    A ~ U(-1/sqrt(in), 1/sqrt(in)), B = 0 (same generator order as the oracle, so seeds are comparable);
  * transformers ``ForCausalLMLoss``: shift by one, ignore_index -100 (the ``input`` part of a record and every patch row
    of a series carry -100), fp32 cross entropy, mean over the counted positions of the optimisation step;
  * ``clip_grad_norm_`` + ``torch.optim.AdamW`` on fp32 master adapters; gradients are summed across the data-parallel
    ranks with ONE all-reduce of the flat gradient arena (NCCL on the GPUs, gloo in the CPU tests).

B200-first layout (DESIGN.md section 7):
  * every matrix product is ``cts_gemm`` (tcgen05): the frozen projections, their input gradients dX = dY W through
    TRANSPOSED copies of the frozen weights that stay resident in HBM (8B: +15 GB of the 180 GB), and the LoRA products,
    which are fused per projection GROUP -- qkv / o / gate_up / down -- into two small GEMMs: U = X A_f^T with the member
    A's stacked ([R, K], R = r x members) and Y += U B_f^T with the member B's block-placed in [N, R] (alpha/r folded in);
  * the skinny weight gradients dB = s dY^T U and dA = dU^T X stream dY / X once (``cts_lora_wgrad``, HBM-bound) straight
    into a flat fp32 gradient arena laid out in peft's parameter shapes, so clip, AdamW and the DP all-reduce are one launch
    / one collective each;
  * all activations of a micro-batch stay resident (no recomputation pass except inside the attention backward):
    ~140 KB per token and layer at the 8B shape, 41 GB for 8192 tokens.

Only ``_cabi.Context`` methods touch numbers; torch allocates, copies and all-reduces.
"""
import json
import math
import os
import re
from dataclasses import dataclass

import numpy as np
import torch

from .trace import span
from ._cabi import EPI_NONE, EPI_RESIDUAL, PACK_DESC_LONGS

TARGETS = ("q_proj", "k_proj", "v_proj", "o_proj", "gate_proj", "up_proj", "down_proj")
IGNORE_INDEX = -100


def _module_of(proj):
    return "self_attn" if proj in ("q_proj", "k_proj", "v_proj", "o_proj") else "mlp"


def _ceil8(n):
    return (n + 7) // 8 * 8


@dataclass
class _Member:
    proj: str          # q_proj ...
    j0: int            # first rank column inside the fused group
    n0: int            # first output row inside the fused weight (plain layout)
    il: int            # 0 plain; 1 gate / 2 up rows of the interleaved gate_up layout
    fin: int           # in features
    fout: int          # out features


class _Group:
    """One fused projection (qkv | o | gu | d) of one layer: the member adapters and their packed operands."""

    def __init__(self, key, K, N, members):
        self.key, self.K, self.N, self.members = key, K, N, members
        self.R = 0          # padded fused rank (multiple of 8: 16-byte rows for TMA)
        self.a_off = 0      # arena offset of the members' stacked A matrices
        self.A = self.At = self.B = self.Bt = None      # views into the work arena


class LoraTrainer:
    def __init__(self, model, r=16, lora_alpha=32, target_modules=TARGETS, lr=1e-4, betas=(0.9, 0.999), eps=1e-8,
                 weight_decay=0.0, max_grad_norm=1.0, seed=0, init_b_std=0.0, group=None, adapters=None):
        if model.tp_size != 1:
            raise ValueError("LoraTrainer is data parallel: build the model with tp_size=1 on every rank")
        if getattr(model, "w4_only", False):
            raise ValueError("LoraTrainer needs the dense projection weights: this model keeps its projections as 4-bit weights only (w4_only)")
        if not 1 <= int(r) <= 64:
            raise ValueError("LoRA rank must be in [1, 64]")
        self.model, self.ctx = model, model.ctx
        self.r, self.alpha = int(r), float(lora_alpha)
        self.scaling = self.alpha / self.r
        self.targets = tuple(t for t in TARGETS if t in set(target_modules))
        if not self.targets:
            raise ValueError(f"target_modules must name some of {TARGETS}")
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        self.max_grad_norm = float(max_grad_norm) if max_grad_norm else 0.0
        self.group = group
        self.step_count = 0
        m = model
        dev, dt = m.device, m.dtype
        self.H, self.I, self.nh, self.nkv, self.d, self.L = m.H, m.I, m.nh, m.nkv, m.d, m.L
        self.QKV = (self.nh + 2 * self.nkv) * self.d
        # ---- frozen weights, transposed once: dX = dY W is then a K-major "TN" GEMM like the forward
        self.wqkv_t = [w.t().contiguous() for w in m.wqkv]          # [H, QKV]
        self.wo_t = [w.t().contiguous() for w in m.wo]              # [nh*d, H]
        self.wgu_t = [w.t().contiguous() for w in m.wgu]            # [H, 2I] (columns in the interleaved order of dgu)
        self.wd_t = [w.t().contiguous() for w in m.wd]              # [I, H]
        self.lm_head_t = m.lm_head.t().contiguous()                 # [H, V]
        # ---- adapter table (peft names and shapes), flat fp32 arenas
        self.index = {}          # name -> (offset, shape)
        off = 0
        self.groups = []         # per layer: dict key -> _Group
        nhd, nkvd = self.nh * self.d, self.nkv * self.d
        spec = {
            "qkv": (self.H, self.QKV, [("q_proj", 0, 0, self.H, nhd), ("k_proj", nhd, 0, self.H, nkvd),
                                       ("v_proj", nhd + nkvd, 0, self.H, nkvd)]),
            "o": (nhd, self.H, [("o_proj", 0, 0, nhd, self.H)]),
            "gu": (self.H, 2 * self.I, [("gate_proj", 0, 1, self.H, self.I), ("up_proj", 0, 2, self.H, self.I)]),
            "d": (self.I, self.H, [("down_proj", 0, 0, self.I, self.H)]),
        }
        for l in range(self.L):
            gl = {}
            for key, (K, N, mem) in spec.items():
                present = [mm for mm in mem if mm[0] in self.targets]
                if not present:
                    continue
                members = [_Member(mm[0], j * self.r, mm[1], mm[2], mm[3], mm[4]) for j, mm in enumerate(present)]
                g = _Group(key, K, N, members)
                g.R = _ceil8(self.r * len(members))
                # arena layout of a group: the members' A matrices STACKED ([r x members, in], contiguous -> their weight gradient
                # is one cts_lora_wgrad launch over the shared input X), then the members' B matrices
                g.a_off = off
                for mm in members:
                    self.index[f"model.layers.{l}.{_module_of(mm.proj)}.{mm.proj}.lora_A.weight"] = (off, (self.r, mm.fin))
                    off += self.r * mm.fin
                for mm in members:
                    self.index[f"model.layers.{l}.{_module_of(mm.proj)}.{mm.proj}.lora_B.weight"] = (off, (mm.fout, self.r))
                    off += mm.fout * self.r
                gl[key] = g
            self.groups.append(gl)
        self.n_params = off
        self.p = torch.zeros(off, device=dev, dtype=torch.float32)
        self.g = torch.zeros(off, device=dev, dtype=torch.float32)
        self.m = torch.zeros(off, device=dev, dtype=torch.float32)
        self.v = torch.zeros(off, device=dev, dtype=torch.float32)
        self.norm_ws = torch.zeros(self.ctx.grad_norm_ws_floats(), device=dev, dtype=torch.float32)
        self.norm_out = torch.zeros(2, device=dev, dtype=torch.float32)          # {||g||, clip coefficient}
        self.loss_out = torch.zeros(1, device=dev, dtype=torch.float32)
        # ---- model-dtype fused operands (work arena) + pack descriptors
        woff = 0
        for gl in self.groups:
            for g in gl.values():
                for name, n in (("A", g.R * g.K), ("At", g.K * g.R), ("B", g.N * g.R), ("Bt", g.R * g.N)):
                    setattr(g, "_off_" + name, woff)
                    woff += _ceil8(n)
        self.work = torch.zeros(max(woff, 8), device=dev, dtype=dt)              # zero blocks / rank padding stay zero for ever
        desc = []
        self.max_pack = 1
        sbits = int(np.float32(self.scaling).view(np.uint32))
        one = int(np.float32(1.0).view(np.uint32))
        for l, gl in enumerate(self.groups):
            for g in gl.values():
                g.A = self.work[g._off_A: g._off_A + g.R * g.K].view(g.R, g.K)
                g.At = self.work[g._off_At: g._off_At + g.K * g.R].view(g.K, g.R)
                g.B = self.work[g._off_B: g._off_B + g.N * g.R].view(g.N, g.R)
                g.Bt = self.work[g._off_Bt: g._off_Bt + g.R * g.N].view(g.R, g.N)
                for mm in g.members:
                    base = f"model.layers.{l}.{_module_of(mm.proj)}.{mm.proj}"
                    oa, _ = self.index[base + ".lora_A.weight"]
                    ob, _ = self.index[base + ".lora_B.weight"]
                    # A [r, in] -> rows [j0, j0+r) of A_f [R, K]; transposed into At_f [K, R]
                    desc.append([oa, self.r, mm.fin, g._off_A, g.K, mm.j0, 0, 0, g._off_At, g.R, one, 0])
                    # B [out, r] -> rows rowmap(i), columns [j0, j0+r) of B_f [N, R] (x alpha/r); transposed into Bt_f [R, N]
                    desc.append([ob, mm.fout, self.r, g._off_B, g.R, mm.n0, mm.il, mm.j0, g._off_Bt, g.N, sbits, 0])
                    self.max_pack = max(self.max_pack, self.r * mm.fin, mm.fout * self.r)
        assert all(len(d) == PACK_DESC_LONGS for d in desc)
        self.n_desc = len(desc)
        self.desc = torch.tensor(desc, dtype=torch.int64).reshape(-1).to(dev)
        # ---- init (peft: A kaiming_uniform(a=sqrt(5)) == U(+-1/sqrt(in)), B zeros), same generator order as oracle/lora.py
        if adapters is None:
            gen = torch.Generator().manual_seed(int(seed))
            host = torch.zeros(off, dtype=torch.float32)
            for l in range(self.L):
                for p in self.targets:
                    base = f"model.layers.{l}.{_module_of(p)}.{p}"
                    oa, sa = self.index[base + ".lora_A.weight"]
                    ob, sb = self.index[base + ".lora_B.weight"]
                    bound = 1.0 / math.sqrt(sa[1])
                    host[oa: oa + sa[0] * sa[1]] = ((torch.rand(sa, generator=gen) * 2 - 1) * bound).reshape(-1)
                    if init_b_std > 0:
                        host[ob: ob + sb[0] * sb[1]] = (torch.randn(sb, generator=gen) * init_b_std).reshape(-1)
            self.p.copy_(host)
        else:
            self.load_adapters(adapters)
        self.pack()

    # ------------------------------------------------------------------------------------------ adapters
    def param(self, name):
        off, shape = self.index[name]
        return self.p[off: off + shape[0] * shape[1]].view(shape)

    def grad(self, name):
        off, shape = self.index[name]
        return self.g[off: off + shape[0] * shape[1]].view(shape)

    def adapters(self):
        """name -> fp32 tensor (clone), peft names without the ``base_model.model.`` prefix."""
        return {n: self.param(n).detach().clone() for n in self.index}

    def grads(self):
        return {n: self.grad(n).detach().clone() for n in self.index}

    def load_adapters(self, sd):
        seen = 0
        for name, t in sd.items():
            mt = re.search(r"(model\.layers\.\d+\.(?:self_attn|mlp)\.\w+_proj\.lora_[AB])(?:\.\w+)?\.weight$", name)
            if not mt:
                continue
            key = mt.group(1) + ".weight"
            if key not in self.index:
                continue
            dst = self.param(key)
            if tuple(t.shape) != tuple(dst.shape):
                raise ValueError(f"{name}: shape {tuple(t.shape)} != {tuple(dst.shape)}")
            dst.copy_(t.to(torch.float32))
            seen += 1
        if seen != len(self.index):
            raise ValueError(f"adapter state holds {seen} of the {len(self.index)} LoRA tensors of this configuration")
        self.pack()

    def save_adapter(self, path):
        """peft layout: adapter_model.safetensors + adapter_config.json (loadable by ChatTSForCausalLM.merge_lora and by
        PeftModel.from_pretrained, demo/demo_lora.ipynb cell 3)."""
        from safetensors.torch import save_file
        os.makedirs(path, exist_ok=True)
        sd = {"base_model.model." + n: self.param(n).detach().cpu().contiguous() for n in self.index}
        save_file(sd, os.path.join(path, "adapter_model.safetensors"))
        cfg = dict(peft_type="LORA", task_type="CAUSAL_LM", r=self.r, lora_alpha=self.alpha, lora_dropout=0.0, bias="none",
                   target_modules=list(self.targets), fan_in_fan_out=False, inference_mode=True)
        with open(os.path.join(path, "adapter_config.json"), "w") as f:
            json.dump(cfg, f, indent=1)

    def pack(self):
        """fp32 master adapters -> the model-dtype fused operands (and their transposes) the GEMMs read."""
        if self.n_desc:
            self.ctx.lora_pack(self.p, self.desc, self.n_desc, self.max_pack, self.work)

    # ------------------------------------------------------------------------------------------ batch preparation
    def _prepare(self, input_ids, attention_mask, timeseries, labels):
        """Host side: merged layout (model._prepare_inputs), labels carried to the merged positions (patch rows: -100),
        the shifted label rows.  Returns a namespace of host arrays; nothing is launched for the decoder yet."""
        m = self.model
        ids_cpu, am_cpu, counts, lay = m._prepare_inputs(input_ids, attention_mask, timeseries)
        lab = torch.as_tensor(labels).cpu().numpy()
        if lab.ndim == 1:
            lab = lab[None]
        if lab.shape != ids_cpu.shape:
            raise ValueError(f"labels {lab.shape} must match input_ids {ids_cpu.shape}")
        B = lay.cu_seqlens.shape[0] - 1
        lens = lay.lens
        sample = np.repeat(np.arange(B), lens)
        merged = np.full(lay.total, IGNORE_INDEX, dtype=np.int64)
        text = lay.src_col >= 0
        merged[text] = lab[sample[text], lay.src_col[text]]
        # ForCausalLMLoss: position i predicts label i+1 of the same sample
        nxt = np.full(lay.total, IGNORE_INDEX, dtype=np.int64)
        nxt[:-1] = merged[1:]
        last = lay.cu_seqlens[1:] - 1
        nxt[last[last >= 0]] = IGNORE_INDEX
        sel = np.nonzero(nxt != IGNORE_INDEX)[0].astype(np.int32)
        ns = type("Batch", (), {})()
        ns.lay, ns.counts, ns.timeseries, ns.host_counts = lay, counts, timeseries, getattr(m, "_host_counts", None)
        ns.sel, ns.targets, ns.n_counted = sel, nxt[sel].astype(np.int32), int(sel.shape[0])
        ns.T, ns.B, ns.max_len = lay.total, B, int(lens.max()) if B else 0
        if ns.max_len > m.n_pos:
            raise ValueError(f"sample of {ns.max_len} positions exceeds max_seq_len {m.n_pos}")
        return ns

    @staticmethod
    def count_labels(batch):
        """Counted label positions of a micro-batch dict, from the labels alone: every real token but the first of its
        sample has exactly one predecessor in the merged sequence (a text token or the last patch row of a series), and
        patch rows never carry a label -- so the count needs neither the series nor the layout."""
        lab = torch.as_tensor(batch["labels"]).cpu().numpy()
        if lab.ndim == 1:
            lab = lab[None]
        am = batch.get("attention_mask")
        am = np.ones_like(lab) if am is None else torch.as_tensor(am).cpu().numpy().reshape(lab.shape)
        n = 0
        for b in range(lab.shape[0]):
            y = lab[b][am[b].astype(bool)]
            n += int((y[1:] != IGNORE_INDEX).sum())
        return n

    # ------------------------------------------------------------------------------------------ forward + backward
    def _lora_fwd(self, g, x, y, T):
        """y += (x A_f^T) B_f^T  (alpha/r folded into B_f); returns U [T, R] for the backward."""
        c = self.ctx
        u = torch.empty(T, g.R, device=x.device, dtype=x.dtype)
        c.gemm(x, g.A, u, epilogue=EPI_NONE, t=T)
        c.gemm(u, g.B, y, residual=y, epilogue=EPI_RESIDUAL, t=T)
        return u

    def _lora_bwd(self, l, g, x, u, dy, dx, T):
        """dU = dY B_f; weight gradients of every member into the arena; dx += dU A_f (when dx is given)."""
        c = self.ctx
        du = torch.empty(T, g.R, device=dy.device, dtype=dy.dtype)
        c.gemm(dy, g.Bt, du, epilogue=EPI_NONE, t=T)
        for mm in g.members:
            gB = self.grad(f"model.layers.{l}.{_module_of(mm.proj)}.{mm.proj}.lora_B.weight")
            c.lora_wgrad(dy, mm.n0, mm.il, mm.fout, u, mm.j0, self.r, T, self.scaling, gB, self.r, 1)        # dB = s dY^T U
        # dA of ALL members in one launch: they share X, their A's are stacked in the arena exactly like dU's columns
        rt, fin = self.r * len(g.members), g.members[0].fin
        if rt <= 64:
            c.lora_wgrad(x, 0, 0, fin, du, 0, rt, T, 1.0, self.g[g.a_off: g.a_off + rt * fin], 1, fin)       # dA = dU^T X
        else:                                                     # cts_lora_wgrad takes at most 64 rank columns per launch
            for mm in g.members:
                gA = self.grad(f"model.layers.{l}.{_module_of(mm.proj)}.{mm.proj}.lora_A.weight")
                c.lora_wgrad(x, 0, 0, mm.fin, du, mm.j0, self.r, T, 1.0, gA, 1, mm.fin)
        if dx is not None:
            c.gemm(du, g.At, dx, residual=dx, epilogue=EPI_RESIDUAL, t=T)

    def forward_backward(self, input_ids, attention_mask=None, timeseries=None, labels=None, denominator=None,
                         accumulate_loss=False, backward=True):
        """One micro-batch: loss contribution (added into self.loss_out) and, when ``backward``, adapter gradients ADDED
        into the arena.  ``denominator`` = counted label positions of the whole optimisation step (default: this batch)."""
        m, c = self.model, self.ctx
        bt = self._prepare(input_ids, attention_mask, timeseries, labels)
        if not accumulate_loss:
            self.loss_out.zero_()
        if bt.n_counted == 0:
            return bt
        dev, dt = m.device, m.dtype
        T, B, lay = bt.T, bt.B, bt.lay
        H, I, nh, nkv, d, QKV, eps = self.H, self.I, self.nh, self.nkv, self.d, self.QKV, m.eps
        denom = float(denominator if denominator else bt.n_counted)
        # inverse of the row selection (scatter of d hidden back to the T positions)
        inv = np.full(T, -1, dtype=np.int32)
        inv[bt.sel] = np.arange(bt.n_counted, dtype=np.int32)
        host = np.concatenate([lay.ids, lay.positions, lay.cu_seqlens, bt.sel, bt.targets, inv]).astype(np.int32)
        dbuf = torch.from_numpy(host).pin_memory().to(dev, non_blocking=True)
        o0 = 0
        ids_d = dbuf[o0: o0 + T]; o0 += T
        pos_d = dbuf[o0: o0 + T]; o0 += T
        cu_d = dbuf[o0: o0 + B + 1]; o0 += B + 1
        sel_d = dbuf[o0: o0 + bt.n_counted]; o0 += bt.n_counted
        tgt_d = dbuf[o0: o0 + bt.n_counted]; o0 += bt.n_counted
        inv_d = dbuf[o0: o0 + T]
        new = lambda *shape, dtype=dt: torch.empty(*shape, device=dev, dtype=dtype)
        # ---- frozen front end: token embeddings + TS patch rows (the TS encoder takes no gradient)
        h = new(T, H)
        c.embed_gather(m.embed, ids_d, h, t=T)
        if bt.counts is not None and lay.row_map.shape[0] > 0:
            rmap = torch.from_numpy(lay.row_map).to(dev, non_blocking=True)
            m.ts_encoder.encode(bt.timeseries, out=h, row_map=rmap, counts=bt.counts, host_counts=bt.host_counts)
        scale = 1.0 / math.sqrt(d)
        saved = []
        # ---------------------------------------------------------------- forward (activations kept for the backward)
        for l in range(self.L):
            gl, s = self.groups[l], {}
            s["h_in"] = h
            xn1 = new(T, H)
            c.reduce_residual_rmsnorm(None, 0, h, None, m.ln1[l], eps, xn1, t=T)
            qkv = new(T, QKV)
            c.gemm(xn1, m.wqkv[l], qkv, bias=m.bqkv[l], epilogue=EPI_NONE, t=T)
            if "qkv" in gl:
                s["u_qkv"] = self._lora_fwd(gl["qkv"], xn1, qkv, T)
            q, k, v = new(T, nh * d), new(T, nkv * d), new(T, nkv * d)
            c.qkv_rope_cache(qkv, False, 1, None, pos_d, m.cos, m.sin, None, q, None, None, k, v, T, nh, nkv, d, m.page_size,
                             m.qn[l], m.kn[l], eps)
            ao, lse = new(T, nh * d), new(T, nh, dtype=torch.float32)
            c.attn_prefill_lse(q, k, v, cu_d, B, bt.max_len, nh, nkv, d, scale, ao, lse)
            h_mid = new(T, H)
            c.gemm(ao, m.wo[l], h_mid, residual=h, epilogue=EPI_RESIDUAL, t=T)
            if "o" in gl:
                s["u_o"] = self._lora_fwd(gl["o"], ao, h_mid, T)
            xn2 = new(T, H)
            c.reduce_residual_rmsnorm(None, 0, h_mid, None, m.ln2[l], eps, xn2, t=T)
            gu = new(T, 2 * I)
            c.gemm(xn2, m.wgu[l], gu, epilogue=EPI_NONE, t=T)
            if "gu" in gl:
                s["u_gu"] = self._lora_fwd(gl["gu"], xn2, gu, T)
            act = new(T, I)
            c.swiglu(gu, T, I, act, interleaved=True)
            h_out = new(T, H)
            c.gemm(act, m.wd[l], h_out, residual=h_mid, epilogue=EPI_RESIDUAL, t=T)
            if "d" in gl:
                s["u_d"] = self._lora_fwd(gl["d"], act, h_out, T)
            s.update(xn1=xn1, qkv=qkv, q=q, k=k, v=v, ao=ao, lse=lse, h_mid=h_mid, xn2=xn2, gu=gu, act=act)
            saved.append(s)
            h = h_out
        # ---------------------------------------------------------------- loss over the label rows
        n = bt.n_counted
        xn = new(T, H)
        c.reduce_residual_rmsnorm(None, 0, h, None, m.final_norm, eps, xn, t=T)
        xs = new(n, H)
        c.gather_rows(xn, sel_d, n, xs)
        logits = new(n, m.V)
        c.gemm(xs, m.lm_head, logits, epilogue=EPI_NONE, t=n)
        row_loss = new(n, dtype=torch.float32)
        c.ce_loss_grad(logits, tgt_d, n, 1.0 / denom, row_loss, self.loss_out, accumulate=True)      # logits <- dlogits
        if not backward:
            return bt
        # ---------------------------------------------------------------- backward
        dxs = new(n, H)
        c.gemm(logits, self.lm_head_t, dxs, epilogue=EPI_NONE, t=n)
        del logits
        dxn = new(T, H)
        c.gather_rows(dxs, inv_d, T, dxn)                    # zero rows where no label is predicted
        dh = new(T, H)
        c.rmsnorm_bwd(dxn, h, m.final_norm, eps, None, dh, t=T)
        delta_ws = new(T, nh, dtype=torch.float32)
        for l in range(self.L - 1, -1, -1):
            gl, s = self.groups[l], saved[l]
            # ---- MLP block: h_out = h_mid + down(act)
            dact = new(T, I)
            c.gemm(dh, self.wd_t[l], dact, epilogue=EPI_NONE, t=T)
            if "d" in gl:
                self._lora_bwd(l, gl["d"], s["act"], s["u_d"], dh, dact, T)
            dgu = new(T, 2 * I)
            c.swiglu_bwd(s["gu"], dact, T, I, dgu, interleaved=True)
            dxn2 = new(T, H)
            c.gemm(dgu, self.wgu_t[l], dxn2, epilogue=EPI_NONE, t=T)
            if "gu" in gl:
                self._lora_bwd(l, gl["gu"], s["xn2"], s["u_gu"], dgu, dxn2, T)
            c.rmsnorm_bwd(dxn2, s["h_mid"], m.ln2[l], eps, dh, dh, t=T)          # dh <- d h_mid (residual + norm path)
            # ---- attention block: h_mid = h_in + o(attn(qkv(norm(h_in))))
            dao = new(T, nh * d)
            c.gemm(dh, self.wo_t[l], dao, epilogue=EPI_NONE, t=T)
            if "o" in gl:
                self._lora_bwd(l, gl["o"], s["ao"], s["u_o"], dh, dao, T)
            dq, dk, dv = new(T, nh * d), new(T, nkv * d), new(T, nkv * d)
            c.attn_bwd(s["q"], s["k"], s["v"], s["ao"], dao, s["lse"], cu_d, B, bt.max_len, nh, nkv, d, scale, delta_ws, dq, dk, dv)
            dqkv = new(T, QKV)
            c.qkv_rope_bwd(dq, dk, dv, s["qkv"], pos_d, m.cos, m.sin, m.qn[l], m.kn[l], eps, dqkv, T, nh, nkv, d)
            if l > 0:
                dxn1 = new(T, H)
                c.gemm(dqkv, self.wqkv_t[l], dxn1, epilogue=EPI_NONE, t=T)
                if "qkv" in gl:
                    self._lora_bwd(l, gl["qkv"], s["xn1"], s["u_qkv"], dqkv, dxn1, T)
                c.rmsnorm_bwd(dxn1, s["h_in"], m.ln1[l], eps, dh, dh, t=T)
            elif "qkv" in gl:
                self._lora_bwd(l, gl["qkv"], s["xn1"], s["u_qkv"], dqkv, None, T)     # the embeddings take no gradient
            saved[l] = None
        return bt

    # ------------------------------------------------------------------------------------------ optimisation step
    def zero_grad(self):
        self.g.zero_()

    def _world(self):
        import torch.distributed as dist
        if self.group is not None or (dist.is_available() and dist.is_initialized()):
            return dist.get_world_size(self.group)
        return 1

    def optimizer_step(self):
        c = self.ctx
        self.step_count += 1
        c.grad_norm_clip(self.g, self.max_grad_norm, self.norm_ws, self.norm_out)
        c.adamw(self.p, self.g, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps, self.weight_decay, self.step_count,
                grad_scale=self.norm_out[1:2])
        self.pack()

    def train_step(self, batches):
        """One optimisation step over ``batches`` (a dict or a list of micro-batch dicts with input_ids, attention_mask,
        timeseries, labels).  Loss = sum of token losses / counted label positions of ALL micro-batches on ALL ranks
        (token-mean over the global batch, what the oracle computes on the union); gradients are summed over the ranks by
        one all-reduce of the arena.  Returns the loss as a 1-element device tensor (read it with .item() when needed)."""
        import torch.distributed as dist
        if isinstance(batches, dict):
            batches = [batches]
        world = self._world()
        local = sum(self.count_labels(b) for b in batches)
        total = local
        if world > 1:
            cnt = torch.tensor([local], dtype=torch.int64, device=self.model.device if dist.get_backend(self.group) == "nccl" else "cpu")
            dist.all_reduce(cnt, group=self.group)
            total = int(cnt.item())
        self.zero_grad()
        self.loss_out.zero_()
        if total > 0:
            for b in batches:
                with span("cts.train.forward_backward"):
                    self.forward_backward(b["input_ids"], b.get("attention_mask"), b.get("timeseries"), b["labels"], denominator=total,
                                          accumulate_loss=True)
        if world > 1:
            with span("cts.train.allreduce"):
                dist.all_reduce(self.g, group=self.group)                # ONE bucket: the whole gradient arena
                dist.all_reduce(self.loss_out, group=self.group)
        with span("cts.train.optimizer"):
            self.optimizer_step()
        return self.loss_out.clone()

    # ------------------------------------------------------------------------------------------ schedule, resume, epochs
    def set_lr(self, lr):
        self.lr = float(lr)

    def state_dict(self):
        """Everything a resumed run needs: master adapters, Adam moments, step counter, hyper-parameters (host tensors)."""
        return {"p": self.p.detach().cpu().clone(), "m": self.m.detach().cpu().clone(), "v": self.v.detach().cpu().clone(),
                "step": self.step_count, "r": self.r, "lora_alpha": self.alpha, "targets": list(self.targets), "n_params": self.n_params,
                "lr": self.lr, "betas": list(self.betas), "eps": self.eps, "weight_decay": self.weight_decay,
                "max_grad_norm": self.max_grad_norm}

    def load_state_dict(self, sd):
        if (sd["r"], list(sd["targets"]), sd["n_params"]) != (self.r, list(self.targets), self.n_params):
            raise ValueError("checkpoint was written for a different LoRA configuration (rank / target modules / model shape)")
        for name in ("p", "m", "v"):
            getattr(self, name).copy_(sd[name])
        self.step_count = int(sd["step"])
        self.lr = float(sd.get("lr", self.lr))
        self.pack()

    def save_checkpoint(self, path):
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        tmp = path + ".tmp"
        torch.save(self.state_dict(), tmp)
        os.replace(tmp, path)                                   # atomic: a killed run never leaves a torn checkpoint

    def load_checkpoint(self, path):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=False))

    def fit(self, processor, records, epochs=1, samples_per_step=8, micro_batch=None, lr_schedule="cosine", warmup_steps=0,
            min_lr_ratio=0.0, eos_token_id=None, max_length=None, shuffle_seed=0, on_step=None, checkpoint=None, checkpoint_every=0):
        """The loop of the external recipe around train_step: every rank walks ITS shard of ``records`` (rank::world) in the
        same seeded order, ``samples_per_step`` records per rank and optimisation step in micro-batches of ``micro_batch``
        (gradient accumulation), learning rate warmed up linearly then decayed (cosine | linear | constant).
        ``checkpoint``: file to resume from if present and to write every ``checkpoint_every`` steps (rank 0 writes)."""
        import torch.distributed as dist
        world = self._world()
        rank = dist.get_rank(self.group) if world > 1 else 0
        mine = shard_records(list(records), rank, world)
        per = max(1, int(samples_per_step))
        steps_per_epoch = len(shard_records(list(records), world - 1, world)) // per        # the shortest shard sets the pace
        if steps_per_epoch == 0:
            raise ValueError(f"{len(records)} records are too few for {world} ranks x {per} samples per step")
        total_steps = steps_per_epoch * int(epochs)
        base_lr = self.lr
        start = 0
        if checkpoint and os.path.exists(checkpoint):
            self.load_checkpoint(checkpoint)
            start = self.step_count
        mb = int(micro_batch or per)
        losses = []
        for step in range(start, total_steps):
            ep, k = divmod(step, steps_per_epoch)
            order = np.random.default_rng(shuffle_seed + ep).permutation(len(mine))
            chunk = [mine[i] for i in order[k * per:(k + 1) * per]]
            self.lr = base_lr * lr_factor(step, total_steps, warmup_steps, lr_schedule, min_lr_ratio)
            batches = [encode_records(processor, chunk[i: i + mb], eos_token_id=eos_token_id, max_length=max_length)
                       for i in range(0, len(chunk), mb)]
            loss = self.train_step(batches)
            losses.append(loss)
            if on_step is not None:
                on_step(step, loss, self)
            if checkpoint and checkpoint_every and (step + 1) % checkpoint_every == 0 and rank == 0:
                self.save_checkpoint(checkpoint)
        self.lr = base_lr
        return [float(l[0]) for l in losses]                                             # one host read at the end

    @torch.no_grad()
    def eval_loss(self, batch):
        self.forward_backward(batch["input_ids"], batch.get("attention_mask"), batch.get("timeseries"), batch["labels"], backward=False)
        return self.loss_out.clone()


def lr_factor(step, total_steps, warmup_steps=0, schedule="cosine", min_ratio=0.0):
    """transformers get_{cosine,linear,constant}_schedule_with_warmup as a pure function of the step."""
    if warmup_steps and step < warmup_steps:
        return (step + 1) / float(warmup_steps + 1) if schedule == "constant" else step / float(max(1, warmup_steps))
    if schedule == "constant":
        return 1.0
    prog = (step - warmup_steps) / float(max(1, total_steps - warmup_steps))
    prog = min(max(prog, 0.0), 1.0)
    dec = 0.5 * (1.0 + math.cos(math.pi * prog)) if schedule == "cosine" else 1.0 - prog
    return min_ratio + (1.0 - min_ratio) * dec


# ---------------------------------------------------------------------------------------------- data
def load_jsonl(path):
    """``{"input": str, "output": str, "timeseries": [[...], ...]}`` per line (chatts/align/uts_template_qa.py:127-131)."""
    out = []
    with open(path) as f:
        for line in f:
            line = line.strip()
            if line:
                r = json.loads(line)
                for key in ("input", "output"):
                    if key not in r:
                        raise ValueError(f"record without '{key}': {list(r)}")
                out.append(r)
    return out


def shard_records(records, rank, world):
    """Data parallel: rank r takes records r, r + world, ..."""
    return list(records[rank::world])


def encode_records(processor, records, eos_token_id=None, max_length=None):
    """records -> micro-batch dict.  Text = input + output (+ eos); labels = -100 on the ``input`` part and on padding,
    the token ids on the ``output`` part.  Series are consumed in ``<ts><ts/>`` order across the batch, like the
    inference processor (chatts/utils/inference_tsmllm_deepspeed.py:75-89)."""
    tok = processor.tokenizer
    series = [np.asarray(ts, dtype=np.float64) for r in records for ts in r.get("timeseries", [])]
    encs, prefixes = processor.encode_series(series)
    k, rows = 0, []
    for r in records:
        n = r["input"].count("<ts><ts/>")
        if "<ts><ts/>" in r["output"]:
            raise ValueError("the output text must not contain <ts><ts/>")
        assert k + n <= len(prefixes), "more <ts><ts/> placeholders than time series"
        rendered_in = processor.render_text(r["input"], prefixes[k: k + n])
        k += n
        ids_in = list(tok.encode(rendered_in))
        ids_out = list(tok.encode(r["output"]))
        if eos_token_id is not None:
            ids_out.append(int(eos_token_id))
        ids = ids_in + ids_out
        lab = [IGNORE_INDEX] * len(ids_in) + ids_out
        if max_length is not None and len(ids) > max_length:
            ids, lab = ids[:max_length], lab[:max_length]
        rows.append((ids, lab))
    assert k == len(prefixes), "time series / <ts><ts/> placeholder count mismatch"
    S = max(len(i) for i, _ in rows)
    pad = tok.pad_token_id if getattr(tok, "pad_token_id", None) is not None else 0
    left = getattr(tok, "padding_side", "left") == "left"
    ids = np.full((len(rows), S), pad, dtype=np.int64)
    am = np.zeros((len(rows), S), dtype=np.int64)
    lab = np.full((len(rows), S), IGNORE_INDEX, dtype=np.int64)
    for b, (i, y) in enumerate(rows):
        sl = slice(S - len(i), S) if left else slice(0, len(i))
        ids[b, sl], am[b, sl], lab[b, sl] = i, 1, y
    out = {"input_ids": torch.from_numpy(ids), "attention_mask": torch.from_numpy(am), "labels": torch.from_numpy(lab)}
    out["timeseries"] = processor.pad_series(encs)
    return out
