"""Attention kernels (csrc/attention.cu) against a float64 reference, with AIMED queries.

With random q and k every key carries about 1/n of a row's weight, so a kernel that drops, adds or misplaces one key of a long row moves
the output by O(1/n): inside any tolerance a 16-bit kernel can be held to.  Here keys are random directions (nearly orthogonal in 64 or
128 dimensions) and each query is a multiple of one chosen key, q = a * k[target] / |k[target]|^2, with a such that the target scores
AIM_NATS above zero while the other keys score ~N(0, AIM_NATS^2 / d): the target takes all but a negligible part of the row's weight and
the output is ~v[target].  Dropping, misplacing or leaking one key then moves the output by O(|v|).  Some queries aim at two keys at
once (q in the span of both, equal scores): the row's weight is split between them, so the merge of two tiles or two decode splits is
exercised too.

Targets are chosen where these kernels can go wrong: the diagonal, the first masked key, key 0, the neighbouring packed sequences, the
first and last key of a 64-key tile, the first and last key of each decode split, rows past a sequence's end and pages the page table
lists past it.  Every KV row a kernel must not read holds GARBAGE: large finite values, the keys signed like the sum of the queries, so that
they would win the softmax if they were read (finite: a non-finite value times p = 0 is NaN even in a correct kernel).

Error per (row, head): max_d |o - ref| / max |v| over that head's visible keys.  The rounding points bound it: P is rounded to the 16-bit
type before P.V and O once at the end, at most about two units in the last place of the model dtype (2^-7 bf16, 2^-10 fp16).  BOUND
holds the bound of each (kernel, dtype) at no more than 1.5 x the worst case measured on a B200.  The two test_aimed_*_faults_* tests (CPU)
apply each targeted fault to the reference itself and check that it moves the rows it touches by at least 10 x that bound.
"""
import math
import os

import pytest
import torch

from tests.gpu_util import ctx, record

gpu = pytest.mark.gpu
BF16, FP16 = torch.bfloat16, torch.float16
DTYPES = [pytest.param(BF16, id="bf16"), pytest.param(FP16, id="fp16")]
TILE = 64                   # key tile of all three kernels (the tcgen05 prefill's query tile is 128, the wmma one's 64)
AIM_NATS = 30.0
GARBAGE = 1.0e4
PAD = TILE                  # garbage rows after the last packed sequence
# Per-row error bounds ("tc5": tcgen05 prefill, "wmma": HMMA prefill, "decode": paged TMA decode), ~1.4 x the worst case over this
# file's cases measured on a B200 (power limit 1000 W); the rounding-point estimate is 2^-7 = 7.8e-3 (bf16), 2^-10 = 9.8e-4 (fp16).
#   measured worst:  tc5 4.28e-3 / 6.05e-4,  wmma 3.82e-3 / 4.13e-4,  decode 2.06e-3 / 2.67e-4   (bf16 / fp16)
BOUND = {("tc5", BF16): 6.0e-3, ("tc5", FP16): 8.5e-4,
         ("wmma", BF16): 5.3e-3, ("wmma", FP16): 5.8e-4,
         ("decode", BF16): 2.9e-3, ("decode", FP16): 3.7e-4}
# |lse - ref| in nats (fp32 statistics; the aimed rows have lse ~ AIM_NATS); measured worst 1.54e-5 (bf16), 3.06e-5 (fp16)
LSE_BOUND = {BF16: 2.2e-5, FP16: 4.3e-5}
SM_COUNT = 148
VARLEN = [1, 63, 64, 65, 0, 127, 128, 129, 577]      # a zero-length sequence in the middle (a repeated cu_seqlens entry)


def _dev():
    return "cuda" if torch.cuda.is_available() else "cpu"


# ============================================================================================ float64 reference
def ref_prefill(q, k, v, cu, nh, nkv, scale, seq_fn=None):
    """Causal varlen GQA in float64: q [>=T, nh, d], k/v [>=T, nkv, d] (16-bit, as the kernel gets them), cu the list of offsets.
    -> o [T, nh, d], lse [T, nh] (natural log).  seq_fn(b, s0, L, kk, vv, W) -> (kk, vv, W) may change one sequence's keys, values and
    key multiplicities W [L, keys] (default: the causal 0/1 mask) -- the self-check's faults."""
    T, d, G = cu[-1], q.shape[-1], nh // nkv
    dev = q.device
    qd, kd, vd = q[:T].double(), k[:T].double(), v[:T].double()
    o = torch.zeros(T, nh, d, dtype=torch.float64, device=dev)
    lse = torch.full((T, nh), -math.inf, dtype=torch.float64, device=dev)
    for b in range(len(cu) - 1):
        s0, L = cu[b], cu[b + 1] - cu[b]
        if L == 0:
            continue
        kk, vv = kd[s0:s0 + L], vd[s0:s0 + L]
        W = torch.ones(L, L, dtype=torch.float64, device=dev).tril()
        if seq_fn is not None:
            kk, vv, W = seq_fn(b, s0, L, kk, vv, W)
        logw = W.log()
        rows = max(1, (1 << 25) // (G * kk.shape[0]))
        for h in range(nkv):
            hs = slice(h * G, (h + 1) * G)
            for r0 in range(0, L, rows):
                r1 = min(L, r0 + rows)
                s = torch.einsum("rgd,jd->grj", qd[s0 + r0:s0 + r1, hs], kk[:, h]) * scale + logw[r0:r1]
                lz = torch.logsumexp(s, -1)
                o[s0 + r0:s0 + r1, hs] = torch.einsum("grj,jd->rgd", torch.exp(s - lz[..., None]).nan_to_num(0.0), vv[:, h])
                lse[s0 + r0:s0 + r1, hs] = lz.T
    return o, lse


def ref_decode(q, kc, vc, page_table, seq_lens, page, scale, w_fn=None):
    """One query per sequence against the paged cache, float64.  -> o [B, nh, d], lse [B, nh], vmax [B, nkv] (max |v| of the visible
    keys).  w_fn(b, n) -> multiplicity [n] of each key (default 1) -- the self-check's faults."""
    B, nh, d = q.shape
    nkv = kc.shape[1]
    G = nh // nkv
    dev = q.device
    o = torch.zeros(B, nh, d, dtype=torch.float64, device=dev)
    lse = torch.zeros(B, nh, dtype=torch.float64, device=dev)
    vmax = torch.zeros(B, nkv, dtype=torch.float64, device=dev)
    for b, n in enumerate(seq_lens):
        t = torch.arange(n, device=dev)
        pg = page_table[b].to(dev).long()[t // page]
        kk, vv = kc[pg, :, t % page].double(), vc[pg, :, t % page].double()      # [n, nkv, d]
        W = torch.ones(n, dtype=torch.float64, device=dev) if w_fn is None else w_fn(b, n)
        s = torch.einsum("hgd,jhd->hgj", q[b].double().view(nkv, G, d), kk) * scale + W.log()
        lz = torch.logsumexp(s, -1)
        o[b] = torch.einsum("hgj,jhd->hgd", torch.exp(s - lz[..., None]).nan_to_num(0.0), vv).reshape(nh, d)
        lse[b] = lz.reshape(nh)
        vmax[b] = vv.abs().amax(dim=(0, 2))
    return o, lse, vmax


# ============================================================================================ aimed inputs
def _aim(k1, k2, scale):
    """q (float32) aimed at k1, or at k1 and k2 alike: the q in span{k1, k2} with scale * q.k1 = scale * q.k2 = AIM_NATS.
    k1 / k2 [..., d]; k2 None or NaN rows: no second key."""
    g11 = (k1 * k1).sum(-1, keepdim=True)
    q = k1 / g11
    if k2 is not None:
        g22, g12 = (k2 * k2).sum(-1, keepdim=True), (k1 * k2).sum(-1, keepdim=True)
        det = g11 * g22 - g12 * g12
        pair = ((g22 - g12) * k1 + (g11 - g12) * k2) / det
        q = torch.where(torch.isnan(k2[..., :1]), q, pair)
    return q * (AIM_NATS / scale)


def _garbage_keys(q, nkv):
    """[nkv, d]: GARBAGE with the sign of the sum of the group's normalised queries (q [rows, nh, d])."""
    rows, nh, d = q.shape
    u = (q / q.norm(dim=-1, keepdim=True).clamp_min(1e-30)).view(rows, nkv, nh // nkv, d).sum(dim=(0, 2))
    return GARBAGE * torch.where(u >= 0, 1.0, -1.0)


PF_KINDS = ("diagonal", "next key (masked)", "key 0", "neighbouring sequence (invisible)", "first key of the tile",
            "last key of the previous tile", "pair: last key of the previous tile + diagonal")


def prefill_inputs(lens, nh, nkv, d, scale, dt, seed):
    """Packed q / k / v of T + PAD rows (the PAD rows hold garbage), cu offsets (list), aims long [T, nh, 2] (global key indices, -1: none).
    Row i of a sequence, head h aims at PF_KINDS[(i + h) % 7]."""
    dev = _dev()
    T = sum(lens)
    cu = [0]
    for n in lens:
        cu.append(cu[-1] + n)
    g = torch.Generator().manual_seed(seed)
    k = torch.randn(T + PAD, nkv, d, generator=g).to(dt).to(dev)
    v = torch.randn(T + PAD, nkv, d, generator=g).to(dt).to(dev)
    aims = torch.full((T, nh, 2), -1, dtype=torch.long)
    live = [b for b in range(len(lens)) if lens[b] > 0]
    for pos, b in enumerate(live):
        s0, L = cu[b], lens[b]
        i = torch.arange(L)
        diag = s0 + i
        nxt = torch.where(s0 + i + 1 < T, s0 + i + 1, diag)
        # the neighbouring sequences: the previous one's last key on even rows, the next one's first key on odd rows (either one if
        # the other does not exist, the diagonal if neither does)
        prev_last = cu[live[pos - 1] + 1] - 1 if pos > 0 else -1
        next_first = cu[live[pos + 1]] if pos + 1 < len(live) else -1
        even, odd = (prev_last if prev_last >= 0 else next_first), (next_first if next_first >= 0 else prev_last)
        neigh = torch.where(i % 2 == 0, even, odd)
        neigh = torch.where(neigh >= 0, neigh, diag)
        tile0 = s0 + (i // TILE) * TILE
        prev_tile_last = s0 + ((i // TILE) * TILE - 1).clamp_min(0)
        first = torch.stack([diag, nxt, torch.full_like(i, s0), neigh, tile0, prev_tile_last, prev_tile_last], 1)    # [L, 7]
        second = torch.full_like(first, -1)
        second[:, 6] = torch.where(prev_tile_last != diag, diag, -1)
        kind = (i.view(L, 1) + torch.arange(nh).view(1, nh)) % len(PF_KINDS)                                        # [L, nh]
        aims[s0:s0 + L, :, 0] = first.gather(1, kind)
        aims[s0:s0 + L, :, 1] = second.gather(1, kind)
    aims = aims.to(dev)
    kvh = torch.arange(nh, device=dev) // (nh // nkv)
    kf = k.float()
    k2 = kf[aims[..., 1].clamp_min(0), kvh]
    k2[aims[..., 1] < 0] = math.nan
    q = torch.empty(T + PAD, nh, d, device=dev)
    q[:T] = _aim(kf[aims[..., 0], kvh], k2, scale)
    del k2
    q[T:] = GARBAGE
    k[T:] = _garbage_keys(q[:T], nkv).to(dt)
    v[T:] = GARBAGE
    return q.to(dt), k, v, cu, aims


def prefill_vmax(v, cu):
    """[T, nkv]: max |v| over the keys row i sees (keys 0..i of its sequence)."""
    va = v[:cu[-1]].double().abs().amax(-1)
    out = torch.empty_like(va)
    for a, b in zip(cu[:-1], cu[1:]):
        if b > a:
            out[a:b] = va[a:b].cummax(0).values
    return out


def decode_splits_of_model(batch, nkv, max_ctx):
    """The split count ChatTSForCausalLM._decode_state (model.py) picks for this batch: fill two CTAs per SM with split x kv head x
    batch CTAs, no more splits than 64-key tiles and at most 32."""
    per = max(1, (2 * SM_COUNT) // max(1, batch * nkv))
    return int(max(1, min(per, (max_ctx + TILE - 1) // TILE, 32)))


def split_ranges(n, splits):
    """[(first key, last key)] of the splits that have tiles, cut as the kernel cuts them: tps = ceil(tiles / splits)."""
    tiles = (n + TILE - 1) // TILE
    tps = (tiles + splits - 1) // splits
    return [(s * tps * TILE, min(n, (s + 1) * tps * TILE) - 1) for s in range(splits) if s * tps < tiles]


def decode_targets(n, splits, page, max_pages):
    """-> (fixed, rest, masked).  fixed: single targets, the new row n - 1, the masked rows, row 0; rest: the pairs straddling each split
    boundary and the first and last key of each split; masked: targets past the sequence (they hold real keys, not garbage, and must
    stay invisible) -- a row >= n inside the last tile and the first row of a page the table lists past the sequence."""
    tiles = (n + TILE - 1) // TILE
    need = (n + page - 1) // page
    masked = [n] if n < tiles * TILE else []
    if need < max_pages and need * page not in masked:
        masked.append(need * page)
    fixed = [(n - 1, -1)] + [(m, -1) for m in masked] + ([(0, -1)] if n > 1 else [])
    rng = split_ranges(n, splits)
    rest = [(rng[s][1], rng[s + 1][0]) for s in range(len(rng) - 1)] + [(a, -1) for r in rng for a in r]
    return fixed, rest, masked


def decode_inputs(seq_lens, nh, nkv, d, page, splits, scale, dt, seed, max_pages=None, spare_pages=3):
    """A paged cache full of garbage; each sequence's visible rows and its masked targets hold random keys and values.  The page tables
    are a random permutation of the pool: the unused entries point at garbage pages, spare pages are in no table.
    -> q [B, nh, d], kc / vc [pages, nkv, page, d], page_table int32 [B, max_pages], aims long [B, nh, 2] (token indices, -1: none)."""
    B, G = len(seq_lens), nh // nkv
    if max_pages is None:
        max_pages = max(-(-n // TILE) * TILE // page for n in seq_lens) + 2
    n_pages = B * max_pages + spare_pages
    g = torch.Generator().manual_seed(seed)
    pt = torch.randperm(n_pages, generator=g)[:B * max_pages].view(B, max_pages)
    kc = torch.zeros(n_pages, nkv, page, d)
    vc = torch.full((n_pages, nkv, page, d), GARBAGE)
    written = torch.zeros(n_pages, page, dtype=torch.bool)
    aims = torch.full((B, nh, 2), -1, dtype=torch.long)
    for b, n in enumerate(seq_lens):
        fixed, rest, masked = decode_targets(n, splits, page, max_pages)
        tok = torch.cat([torch.arange(n), torch.tensor(masked, dtype=torch.long)])
        pg, rw = pt[b][tok // page], tok % page
        kc[pg, :, rw] = torch.randn(len(tok), nkv, d, generator=g)
        vc[pg, :, rw] = torch.randn(len(tok), nkv, d, generator=g)
        written[pg, rw] = True
        for x, y in (a for a in rest if a[1] >= 0):            # a pair's two values point opposite ways: its merge moves the output most
            vc[pt[b][y // page], :, y % page] = -vc[pt[b][x // page], :, x % page]
        for h in range(nh):
            if h < len(fixed) or not rest:
                aims[b, h] = torch.tensor(fixed[h % len(fixed)])
            else:
                aims[b, h] = torch.tensor(rest[(h - len(fixed) + b * nh) % len(rest)])
    kc, vc = kc.to(dt).float(), vc.to(dt).float()
    kvh = torch.arange(nh) // G
    q = torch.empty(B, nh, d)
    for b in range(B):
        t1, t2 = aims[b, :, 0], aims[b, :, 1]
        k2 = kc[pt[b][t2.clamp_min(0) // page], kvh, t2.clamp_min(0) % page]
        k2[t2 < 0] = math.nan
        q[b] = _aim(kc[pt[b][t1 // page], kvh, t1 % page], k2, scale)
    gk = _garbage_keys(q, nkv)
    kc = torch.where(written.view(n_pages, 1, page, 1), kc, gk.view(1, nkv, 1, d))
    dev = _dev()
    return q.to(dt).to(dev), kc.to(dt).to(dev), vc.to(dt).to(dev), pt.to(torch.int32).to(dev), aims


def _worst(err):
    """(worst value, row, head) of an error tensor [rows, heads]."""
    r, h = divmod(int(err.argmax()), err.shape[1])
    return float(err[r, h]), r, h


# ============================================================================================ prefill on the GPU
@pytest.fixture(scope="module")
def wmma_ctx():
    """A second context with CTS_ATTN_WMMA=1 (read at context creation): head_dim 128 through the HMMA prefill kernel."""
    from chatts_b200 import _cabi
    old = os.environ.get("CTS_ATTN_WMMA")
    os.environ["CTS_ATTN_WMMA"] = "1"
    try:
        c = _cabi.Context()
    finally:
        if old is None:
            del os.environ["CTS_ATTN_WMMA"]
        else:
            os.environ["CTS_ATTN_WMMA"] = old
    yield c
    torch.cuda.synchronize()
    c.close()


def _prefill_case(request, path, lens, nh, nkv, d, dt, scale=None):
    c = request.getfixturevalue("wmma_ctx") if path == "wmma128" else ctx()
    family = "tc5" if path == "tc5" else "wmma"
    scale = d ** -0.5 if scale is None else scale
    q, k, v, cu, aims = prefill_inputs(lens, nh, nkv, d, scale, dt, seed=sum(lens) + 7 * nh + d + (dt == FP16))
    T, n_rows = cu[-1], cu[-1] + PAD
    cu_t = torch.tensor(cu, dtype=torch.int32).cuda()
    out = torch.full((n_rows, nh * d), math.nan, device="cuda", dtype=dt)
    out_l = torch.full((n_rows, nh * d), math.nan, device="cuda", dtype=dt)
    lse = torch.full((n_rows, nh), math.nan, device="cuda", dtype=torch.float32)
    c.attn_prefill(q, k, v, cu_t, len(lens), max(lens), nh, nkv, d, scale, out)
    c.attn_prefill_lse(q, k, v, cu_t, len(lens), max(lens), nh, nkv, d, scale, out_l, lse)
    torch.cuda.synchronize()
    ref, ref_lse = ref_prefill(q, k, v, cu, nh, nkv, scale)
    vmax = prefill_vmax(v, cu)[:, torch.arange(nh) // (nh // nkv)]
    for o in (out, out_l):
        assert torch.isnan(o[T:].float()).all(), "a row past the last sequence was written"
        assert torch.isfinite(o[:T].float()).all()
    assert torch.isnan(lse[T:]).all()
    err, r, h, entry = max(_worst((o[:T].view(T, nh, d).double() - ref).abs().amax(-1) / vmax) + (entry,)
                           for o, entry in ((out, "cts_attn_prefill"), (out_l, "cts_attn_prefill_lse")))
    lse_err, lr, lh = _worst((lse[:T].double() - ref_lse).abs())
    bound = BOUND[(family, dt)]
    record("attn_aimed_prefill", kernel=path, dtype=str(dt).split(".")[-1], nh=nh, nkv=nkv, d=d, lens=str(lens), scale=scale, err=err,
           lse_err=lse_err, bound=bound, lse_bound=LSE_BOUND[dt])
    assert err <= bound, f"{entry}: row {r} head {h} (aimed at {aims[r, h].tolist()}): {err:.3e} of max|v| (bound {bound:.1e})"
    assert lse_err <= LSE_BOUND[dt], f"row {lr} head {lh}: |lse - ref| = {lse_err:.3e} (bound {LSE_BOUND[dt]:.1e})"


PF_LAYOUTS = [(128, 40, 8), (128, 32, 8), (128, 20, 4), (128, 10, 2), (128, 5, 1), (64, 8, 2), (64, 4, 1)]
PF_PATHS = [pytest.param(d, nh, nkv, p, id=f"{nh}-{nkv}-d{d}-{p}") for d, nh, nkv in PF_LAYOUTS
            for p in (["tc5", "wmma128"] if d == 128 else ["wmma64"])]


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("d,nh,nkv,path", PF_PATHS)
def test_prefill_aimed_varlen(request, d, nh, nkv, path, dt):
    """The model's head layouts and its tensor-parallel shards (40/8, 20/4, 10/2, 5/1), lengths around the 64- and 128-row tiles, a
    zero-length sequence in the middle, garbage after the last sequence; out and lse of both entry points."""
    _prefill_case(request, path, VARLEN, nh, nkv, d, dt)


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("scale", [0.05, 1.0])
@pytest.mark.parametrize("d,nh,nkv,path", [pytest.param(128, 40, 8, "tc5", id="40-8-d128-tc5"),
                                           pytest.param(128, 40, 8, "wmma128", id="40-8-d128-wmma128"),
                                           pytest.param(64, 8, 2, "wmma64", id="8-2-d64-wmma64")])
def test_prefill_aimed_scale(request, d, nh, nkv, path, scale, dt):
    """scale != 1/sqrt(d): the aims are set for the given scale, so a kernel that ignored the argument would miss every target."""
    _prefill_case(request, path, VARLEN, nh, nkv, d, dt, scale=scale)


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("nh,nkv", [(5, 1), (40, 8)])
def test_prefill_aimed_config4(request, nh, nkv, dt):
    """bench.py's config 4 prefill: 8 x 2464 positions."""
    _prefill_case(request, "tc5", [2464] * 8, nh, nkv, 128, dt)


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("path", ["tc5", "wmma128"])
def test_prefill_aimed_4096(request, path, dt):
    _prefill_case(request, path, [4096], 40, 8, 128, dt)


# ============================================================================================ decode on the GPU
def _decode_case(seq_lens, nh, nkv, d, page, splits, dt, max_pages=None):
    c = ctx()
    scale = d ** -0.5
    B = len(seq_lens)
    q, kc, vc, pt, aims = decode_inputs(seq_lens, nh, nkv, d, page, splits, scale, dt, seed=sum(seq_lens) + nh + page + splits,
                                        max_pages=max_pages)
    ref, _, vmax = ref_decode(q, kc, vc, pt, seq_lens, page, scale)
    vmax = vmax[:, torch.arange(nh) // (nh // nkv)]
    sl = torch.tensor(seq_lens, dtype=torch.int32).cuda()
    ws = torch.zeros(c.attn_decode_workspace_floats(B, nh, d, splits), device="cuda", dtype=torch.float32)
    bound = BOUND[("decode", dt)]
    worst = 0.0
    for run in range(2):            # twice on one workspace: the arrival counters must reset themselves
        out = torch.full((B, nh * d), math.nan, device="cuda", dtype=dt)
        c.attn_decode(q, kc, vc, pt, sl, B, nh, nkv, d, page, scale, splits, ws, out)
        torch.cuda.synchronize()
        assert torch.isfinite(out.float()).all()
        err, b, h = _worst((out.view(B, nh, d).double() - ref).abs().amax(-1) / vmax)
        assert err <= bound, (f"run {run}: sequence {b} (seq_len {seq_lens[b]}) head {h}, aimed at {aims[b, h].tolist()}: "
                              f"{err:.3e} of max|v| (bound {bound:.1e})")
        worst = max(worst, err)
        assert (ws[B * nh * splits * (d + 2):] == 0).all(), "arrival counters not reset"
    record("attn_aimed_decode", dtype=str(dt).split(".")[-1], nh=nh, nkv=nkv, d=d, page=page, splits=splits, seq_lens=str(seq_lens),
           err=worst, bound=bound)


DEC_CONTEXTS = [1, 64, 65, 2464, 4097]
DEC_TILES = (max(DEC_CONTEXTS) + TILE - 1) // TILE


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("splits", ["1", "model", "32", "more_than_tiles"])
@pytest.mark.parametrize("page", [16, 32, 64])
@pytest.mark.parametrize("d,nh,nkv", [pytest.param(128, 40, 8, id="40-8-d128"), pytest.param(128, 5, 1, id="5-1-d128"),
                                      pytest.param(64, 8, 2, id="8-2-d64")])
def test_decode_aimed(d, nh, nkv, page, splits, dt):
    """Contexts 1 .. 4097 in one batch: heads aim at the new row, row 0, the first and last key of every split, pairs across split
    boundaries, a masked row of the last tile and a page listed past the sequence; page tables scattered over a pool of garbage."""
    n = {"1": 1, "model": decode_splits_of_model(len(DEC_CONTEXTS), nkv, max(DEC_CONTEXTS)), "32": 32,
         "more_than_tiles": DEC_TILES + 3}[splits]
    _decode_case(DEC_CONTEXTS, nh, nkv, d, page, n, dt)


@gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("spare_entries", [0, 2])
def test_decode_aimed_page_ids_past_shared_memory(spare_entries, dt):
    """A CTA keeps at most 256 page ids in shared memory and reads the rest of its page table from global memory.  Batch 32 x 8 kv
    heads runs one split (the model's heuristic), so with 16-token pages any context above 4096 takes this path; here 66 tiles x 4
    pages = 264 page ids per CTA, and with spare_entries = 0 the table is exactly as wide as the last tile (its clamp is exercised)."""
    assert decode_splits_of_model(32, 8, 4224) == 1
    seq_lens, page = [4163, 4224], 16
    for n in seq_lens:
        assert (n + TILE - 1) // TILE * (TILE // page) > 256            # ntl * npp of the single split
    _decode_case(seq_lens, 40, 8, 128, page, 1, dt, max_pages=4224 // page + spare_entries)


@gpu
def test_decode_sees_the_row_written_by_its_pdl_predecessor():
    """cts_attn_decode loads the KV tiles before the one that holds row seq_len - 1 ahead of its dependency wait.  Its predecessor on
    the stream, cts_qkv_rope_cache, writes row seq_len - 1 (a new key and a distinctive value) and q; the heads aimed at the new key
    must return the new value, not the stale row.  Run once."""
    c = ctx()
    dt, d, nh, nkv, page = BF16, 128, 40, 8, 16
    seq_lens = [2464, 2465, 4097, 65]
    B, G = len(seq_lens), nh // nkv
    splits = decode_splits_of_model(B, nkv, max(seq_lens))
    scale = d ** -0.5
    q, kc, vc, pt, aims = decode_inputs(seq_lens, nh, nkv, d, page, splits, scale, dt, seed=5)
    g = torch.Generator().manual_seed(6)
    k_new = torch.randn(B, nkv, d, generator=g).to(dt).float()
    v_new = (3.0 * torch.randn(B, nkv, d, generator=g)).to(dt)
    new = (aims[:, :, 0] == torch.tensor(seq_lens).view(B, 1) - 1) | (torch.arange(nh) % G == 0).view(1, nh)   # [B, nh]
    kvh = torch.arange(nh) // G
    q_src = q.float().cpu()
    q_src[new] = _aim(k_new[:, kvh][new], None, scale)
    src = torch.cat([q_src.reshape(B, -1), k_new.reshape(B, -1), v_new.float().reshape(B, -1)], 1).to(dt).cuda()
    cos, sin = torch.ones(1, d // 2, dtype=dt).cuda(), torch.zeros(1, d // 2, dtype=dt).cuda()     # position 0: RoPE is the identity
    pos = torch.zeros(B, dtype=torch.int32).cuda()
    new_page = [int(pt[b, (n - 1) // page]) for b, n in enumerate(seq_lens)]
    slot = torch.tensor([p * page + (n - 1) % page for p, n in zip(new_page, seq_lens)], dtype=torch.int32).cuda()
    stale_k = torch.stack([kc[p, :, (n - 1) % page] for p, n in zip(new_page, seq_lens)]).float().cpu()
    assert (stale_k - k_new).abs().amax() > 1.0
    q_out = torch.full((B, nh * d), math.nan, device="cuda", dtype=dt)
    sl = torch.tensor(seq_lens, dtype=torch.int32).cuda()
    ws = torch.zeros(c.attn_decode_workspace_floats(B, nh, d, splits), device="cuda", dtype=torch.float32)
    out = torch.full((B, nh * d), math.nan, device="cuda", dtype=dt)
    c.qkv_rope_cache(src, False, 1, None, pos, cos, sin, slot, q_out, kc, vc, None, None, B, nh, nkv, d, page)
    c.attn_decode(q_out.view(B, nh, d), kc, vc, pt, sl, B, nh, nkv, d, page, scale, splits, ws, out)
    torch.cuda.synchronize()
    assert torch.equal(q_out.cpu().view(B, nh, d), q_src.to(dt))
    for b, (p, n) in enumerate(zip(new_page, seq_lens)):
        assert torch.equal(kc[p, :, (n - 1) % page].float().cpu(), k_new[b])
        assert torch.equal(vc[p, :, (n - 1) % page].cpu(), v_new[b])
    ref, _, vmax = ref_decode(q_out.view(B, nh, d), kc, vc, pt, seq_lens, page, scale)
    vmax = vmax[:, kvh]
    o = out.view(B, nh, d).double()
    bound = BOUND[("decode", dt)]
    err, b, h = _worst((o - ref).abs().amax(-1) / vmax)
    to_new = ((o.cpu() - v_new.double()[:, kvh]).abs().amax(-1) / vmax.cpu())[new]
    record("attn_aimed_decode_pdl", dtype="bfloat16", splits=splits, err=err, err_new_row=float(to_new.max()), bound=bound)
    assert err <= bound, f"sequence {b} head {h}: {err:.3e} of max|v| (bound {bound:.1e})"
    assert float(to_new.max()) <= bound, f"a head aimed at the new row is {float(to_new.max()):.3e} from its value"


# ============================================================================================ sensitivity of the aimed inputs (CPU)
def _report(dt, shifts):
    """Every fault must move each (row, head) it touches by >= 10 x the dtype's largest bound."""
    need = 10 * max(b for (_, t), b in BOUND.items() if t == dt)
    for name, sh in shifts.items():
        assert sh.numel() > 0, f"{name}: no aimed (row, head) is touched by this fault"
        print(f"{str(dt).split('.')[-1]} {name}: moves {sh.numel()} aimed (row, head) pairs by >= {float(sh.min()):.3e} of max|v| "
              f"(must exceed 10 x bound = {need:.3e})")
        assert float(sh.min()) >= need, f"{name}: a touched row moves only {float(sh.min()):.3e} (10 x bound {need:.3e})"


@pytest.mark.parametrize("dt", DTYPES)
def test_aimed_prefill_faults_move_the_reference_past_the_bound(dt):
    """Applies each targeted prefill fault to the float64 reference (at small sizes, same aimed inputs as the GPU tests)."""
    lens, nh, nkv, d = [1, 63, 64, 0, 65, 130, 129], 10, 2, 128
    scale = d ** -0.5
    q, k, v, cu, aims = prefill_inputs(lens, nh, nkv, d, scale, dt, seed=11)
    q, k, v, aims = q.cpu(), k.cpu(), v.cpu(), aims.cpu()
    T = cu[-1]
    ref, _ = ref_prefill(q, k, v, cu, nh, nkv, scale)
    vmax = prefill_vmax(v, cu)[:, torch.arange(nh) // (nh // nkv)]
    kd, vd = k.double(), v.double()
    live = [b for b in range(len(lens)) if lens[b] > 0]
    prev = {b: live[n - 1] for n, b in enumerate(live) if n > 0}
    nxt = {b: live[n + 1] for n, b in enumerate(live) if n + 1 < len(live)}
    seq = torch.repeat_interleave(torch.arange(len(lens)), torch.tensor(lens))
    row = torch.arange(T).view(T, 1, 1)
    s0 = torch.tensor(cu[:-1])[seq].view(T, 1, 1)
    L = torch.tensor(lens)[seq].view(T, 1, 1)
    i, j = row - s0, aims - s0
    inside = (aims >= 0) & (j >= 0) & (j < L)
    visible = inside & (j <= i)
    n_prev = torch.tensor([min(TILE, lens[b], lens[prev[b]]) if b in prev else 0 for b in range(len(lens))])[seq].view(T, 1, 1)
    next0 = torch.tensor([cu[nxt[b]] if b in nxt else -1 for b in range(len(lens))])[seq].view(T, 1, 1)
    n_next = torch.tensor([min(TILE, lens[nxt[b]]) if b in nxt else 0 for b in range(len(lens))])[seq].view(T, 1, 1)

    def remask(f):
        def seq_fn(b, a, n, kk, vv, W):
            return kk, vv, f(torch.arange(n).view(n, 1), torch.arange(n).view(1, n), W)
        return seq_fn

    def previous_first_tile(b, a, n, kk, vv, W):              # a wrong sequence offset: the previous sequence's first tile
        if b not in prev:
            return kk, vv, W
        p, m = cu[prev[b]], min(TILE, n, lens[prev[b]])
        return torch.cat([kd[p:p + m], kk[m:]]), torch.cat([vd[p:p + m], vv[m:]]), W

    def next_first_tile(b, a, n, kk, vv, W):                  # reading on past the end into the next sequence
        if b not in nxt:
            return kk, vv, W
        p, m = cu[nxt[b]], min(TILE, lens[nxt[b]])
        return torch.cat([kk, kd[p:p + m]]), torch.cat([vv, vd[p:p + m]]), torch.cat([W, torch.ones(n, m, dtype=W.dtype)], 1)

    faults = [
        ("drop the diagonal", remask(lambda ii, jj, W: torch.where(jj == ii, 0.0, W)), aims == row),
        ("leak key i + 1", remask(lambda ii, jj, W: torch.where(jj == ii + 1, 1.0, W)), inside & (j == i + 1)),
        ("drop the first key of every tile", remask(lambda ii, jj, W: torch.where(jj % TILE == 0, 0.0, W)), visible & (j % TILE == 0)),
        ("drop the last key of every tile", remask(lambda ii, jj, W: torch.where(jj % TILE == TILE - 1, 0.0, W)),
         visible & (j % TILE == TILE - 1)),
        ("read the previous sequence's first tile instead of its own", previous_first_tile, visible & (j < n_prev)),
        ("read the next sequence's first tile as well", next_first_tile, (aims >= next0) & (aims < next0 + n_next) & (next0 >= 0)),
    ]
    shifts = {}
    for name, seq_fn, touched in faults:
        o, _ = ref_prefill(q, k, v, cu, nh, nkv, scale, seq_fn=seq_fn)
        shifts[name] = ((o - ref).abs().amax(-1) / vmax)[touched.any(-1)]
    _report(dt, shifts)


@pytest.mark.parametrize("dt", DTYPES)
def test_aimed_decode_faults_move_the_reference_past_the_bound(dt):
    """Drops each decode split's key range, or counts it twice (a merge that takes one partial twice), in the float64 reference.
    Counting a range twice moves only rows whose weight straddles it: the pairs aimed across split boundaries."""
    seq_lens, nh, nkv, d, page, splits = [65, 300, 700], 8, 2, 64, 16, 3
    scale = d ** -0.5
    q, kc, vc, pt, aims = decode_inputs(seq_lens, nh, nkv, d, page, splits, scale, dt, seed=12)
    ref, _, vmax = ref_decode(q, kc, vc, pt, seq_lens, page, scale)
    vmax = vmax[:, torch.arange(nh) // (nh // nkv)]
    shifts = {"drop a split's range": [], "count a split's range twice": []}
    for s in range(splits):
        rng = [split_ranges(n, splits) for n in seq_lens]
        lo = torch.tensor([r[s][0] if s < len(r) else -1 for r in rng]).view(-1, 1, 1)
        hi = torch.tensor([r[s][1] if s < len(r) else -2 for r in rng]).view(-1, 1, 1)
        hit = (aims >= lo) & (aims <= hi)
        for name, mult, touched in (("drop a split's range", 0.0, hit.any(-1)),
                                    ("count a split's range twice", 2.0, (hit.sum(-1) == 1) & (aims[..., 1] >= 0))):
            def w_fn(b, n, s=s, mult=mult):
                W = torch.ones(n, dtype=torch.float64)
                r = split_ranges(n, splits)
                if s < len(r):
                    W[r[s][0]:r[s][1] + 1] = mult
                return W
            o, _, _ = ref_decode(q, kc, vc, pt, seq_lens, page, scale, w_fn=w_fn)
            shifts[name].append(((o - ref).abs().amax(-1) / vmax)[touched])
    _report(dt, {k: torch.cat(v) for k, v in shifts.items()})
