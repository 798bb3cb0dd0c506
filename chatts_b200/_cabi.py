"""ctypes binding of libchatts_b200.so (include/chatts_b200.h).

This is the ONLY compute path of the package: there is no Python / torch fallback behind any wrapper, and
importing the package on a machine where the library is missing or where no sm_100 GPU is visible raises
as soon as a kernel is requested.  torch is used for device memory, streams and torch.distributed only.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libchatts_b200.so")

OK = 0
BF16, F16 = 0, 1
EPI_NONE, EPI_GELU, EPI_SWIGLU, EPI_PARTIAL_F32, EPI_RESIDUAL, EPI_SPLITK_F32, EPI_SWIGLU_IL = 0, 1, 2, 3, 4, 5, 6

# every symbol include/chatts_b200.h declares (tests/test_cabi_symbols.py checks the .so exports them all)
SYMBOLS = [
    "cts_version", "cts_arch", "cts_ctx_create", "cts_ctx_destroy", "cts_last_error",
    "cts_ts_patch_count", "cts_ts_patchify", "cts_gemm", "cts_gemm_suggest_split",
    "cts_reduce_bias_act", "cts_reduce_residual_rmsnorm", "cts_reduce_swiglu", "cts_qkv_rope_cache",
    "cts_embed_gather", "cts_attn_prefill", "cts_attn_decode_workspace_floats", "cts_attn_decode",
    "cts_greedy_advance", "cts_ipc_alloc", "cts_ipc_open", "cts_ipc_close", "cts_ipc_free",
    "cts_peer_allreduce_residual_rmsnorm", "cts_peer_greedy_advance", "cts_decode_chain",
    # A9: LoRA fine-tune step
    "cts_attn_prefill_lse", "cts_attn_bwd", "cts_swiglu", "cts_swiglu_bwd", "cts_rmsnorm_bwd", "cts_qkv_rope_bwd",
    "cts_ce_loss_grad", "cts_gather_rows", "cts_lora_wgrad", "cts_adamw", "cts_grad_norm_ws_floats", "cts_grad_norm_clip",
    "cts_lora_pack",
    "cts_sample_advance", "cts_rmsnorm", "cts_lm_head", "cts_decoder_step_ws_floats", "cts_decoder_step", "cts_ts_encode", "cts_gemm_decode_fused",
    "cts_peer_ll_region_bytes", "cts_peer_allreduce_ll", "cts_trace_enable", "cts_ts_encode_fused_ok", "cts_ts_encode_fused",
    "cts_rep_penalty_mark", "cts_rep_penalty_apply", "cts_gemm_w4", "cts_gemm_w4_suggest_split", "cts_gemm_w4_mma", "cts_gemm_w4_mma_suggest_split",
    "cts_gemm_w4_prefill",
]
FUSED_RESIDUAL, FUSED_SWIGLU, FUSED_QKV_ROPE = 0, 1, 2
PACK_DESC_LONGS = 12


class CtsError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("w", C.c_void_p), ("w2", C.c_void_p), ("x", C.c_void_p), ("bias", C.c_void_p),
        ("residual", C.c_void_p), ("out", C.c_void_p), ("row_map", C.c_void_p),
        ("n", C.c_longlong), ("k", C.c_longlong), ("t", C.c_longlong),
        ("w_ld", C.c_longlong), ("x_ld", C.c_longlong), ("out_ld", C.c_longlong),
        ("dtype", C.c_int), ("epilogue", C.c_int), ("split_k", C.c_int), ("reserved", C.c_int),
        ("splitk_ws", C.c_void_p), ("tile_counters", C.c_void_p),
        ("next_w", C.c_void_p), ("next_n", C.c_longlong), ("next_k", C.c_longlong), ("next_ld", C.c_longlong),
        ("next_split", C.c_int), ("next_reserved", C.c_int), ("next_prefetch_bytes", C.c_longlong),
    ]


class ChainArgs(C.Structure):
    _fields_ = (
        [(k, C.c_int) for k in ("t", "hidden", "inter", "nh", "nkv", "head_dim", "phase_begin", "phase_end", "norm5_has_partial",
                                "dtype")] + [("split", C.c_int * 4)] +
        [(k, C.c_void_p) for k in ("wo", "wgu", "wd", "wqkv", "ao", "h", "xn", "act", "ln_post", "ln_next")] + [("eps", C.c_float)] +
        [(k, C.c_void_p) for k in ("bqkv", "q_norm_w", "k_norm_w", "positions", "cos_tab", "sin_tab", "slot_map", "q_out", "k_cache",
                                   "v_cache")] + [("page_size", C.c_int)] + [(k, C.c_void_p) for k in ("ws", "ssq", "sync")])


class LayerWeights(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("wqkv", "bqkv", "q_norm", "k_norm", "wo", "wgu", "wd", "ln1", "ln2", "k_cache", "v_cache")]


class DecoderStepArgs(C.Structure):
    _fields_ = (
        [(k, C.c_int) for k in ("n_layers", "hidden", "inter", "nh", "nkv", "head_dim", "vocab", "vocab_rows", "page_size", "num_pages",
                                "max_pages", "dtype", "batch", "sample")] + [("eps", C.c_float)] +
        [(k, C.c_int) for k in ("split_qkv", "split_o", "split_gu", "split_d", "attn_splits")] +
        [("layers", C.POINTER(LayerWeights))] +
        [(k, C.c_void_p) for k in ("embed", "final_norm", "lm_head", "cos_tab", "sin_tab", "cur_ids", "positions", "seq_lens", "slot_map",
                                   "page_table", "out_tokens")] + [("out_ld", C.c_int)] +
        [(k, C.c_void_p) for k in ("step_ptr", "h", "xn", "q", "ao", "act", "logits", "ws")] + [("ws_floats", C.c_longlong)] +
        [("attn_ws", C.c_void_p)])


class FusedGemmArgs(C.Structure):
    _fields_ = ([("w", C.c_void_p), ("x", C.c_void_p), ("n", C.c_longlong), ("k", C.c_longlong), ("t", C.c_longlong)] +
                [(k, C.c_int) for k in ("dtype", "mode", "split_k", "reserved")] +
                [(k, C.c_void_p) for k in ("bias", "h", "act", "positions", "cos_tab", "sin_tab", "slot_map", "q_out", "k_cache", "v_cache",
                                           "q_norm", "k_norm")] + [("eps", C.c_float)] +
                [(k, C.c_int) for k in ("nh", "nkv", "head_dim", "page_size")] +
                [("norm_h", C.c_void_p), ("norm_w", C.c_void_p), ("ssq_in", C.c_void_p), ("ssq_tiles", C.c_int), ("norm_eps", C.c_float),
                 ("ssq_out", C.c_void_p), ("peer_regions", C.c_void_p), ("peer_state", C.c_void_p)] +
                [(k, C.c_int) for k in ("peer_rank", "peer_world", "peer_max_tokens", "peer_reserved")] + [("peer_region_bytes", C.c_longlong)])


class GemmW4Args(C.Structure):
    _fields_ = [("qw", C.c_void_p), ("scales", C.c_void_p), ("zeros", C.c_void_p), ("x", C.c_void_p), ("out", C.c_void_p),
                ("n", C.c_longlong), ("k", C.c_longlong), ("t", C.c_longlong), ("x_ld", C.c_longlong),
                ("group_size", C.c_int), ("split_k", C.c_int), ("dtype", C.c_int), ("reserved", C.c_int)]


class GemmW4pArgs(C.Structure):
    _fields_ = [("qw", C.c_void_p), ("szp", C.c_void_p), ("x", C.c_void_p), ("bias", C.c_void_p), ("residual", C.c_void_p), ("out", C.c_void_p),
                ("n", C.c_longlong), ("k", C.c_longlong), ("t", C.c_longlong), ("x_ld", C.c_longlong), ("out_ld", C.c_longlong),
                ("group_size", C.c_int), ("split_k", C.c_int), ("dtype", C.c_int), ("epilogue", C.c_int)]


class GemmW4fArgs(C.Structure):
    _fields_ = [("qw", C.c_void_p), ("szp", C.c_void_p), ("x", C.c_void_p), ("out", C.c_void_p),
                ("n", C.c_longlong), ("k", C.c_longlong), ("t", C.c_longlong), ("x_ld", C.c_longlong),
                ("group_size", C.c_int), ("split_k", C.c_int), ("dtype", C.c_int), ("reserved", C.c_int)]


class TsEncodeArgs(C.Structure):
    _fields_ = ([("x", C.c_void_p)] + [(k, C.c_int) for k in ("dtype", "n_series", "row_len", "num_features", "patch_size", "mode")] +
                [("pos_table", C.c_void_p)] + [(k, C.c_int) for k in ("emb_dim", "max_seq_len", "num_layers", "hidden", "in0")] +
                [("weights", C.POINTER(C.c_void_p)), ("biases", C.POINTER(C.c_void_p))] +
                [(k, C.c_void_p) for k in ("valid_len", "patch_cnt", "row_offset", "max_valid")] + [("total_rows", C.c_longlong)] +
                [("rows_ws", C.c_void_p), ("act_ws", C.c_void_p * 2), ("splitk_ws", C.c_void_p), ("splitk_floats", C.c_longlong),
                 ("out", C.c_void_p), ("out_ld", C.c_longlong), ("row_map", C.c_void_p)])


_lib = None


def load_library():
    """dlopen the in-tree library; raise loudly if it is not there (no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CtsError(f"{LIB_PATH} is missing: run `python -m chatts_b200.build` (nvcc, sm_100a). "
                       "chatts_b200 has no CPU or torch fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i, ll, f = C.c_void_p, C.c_int, C.c_longlong, C.c_float
    lib.cts_version.restype = i
    lib.cts_arch.restype = C.c_char_p
    lib.cts_ctx_create.argtypes = [i, C.POINTER(vp)]
    lib.cts_ctx_destroy.argtypes = [vp]
    lib.cts_ctx_destroy.restype = None
    lib.cts_last_error.argtypes = [vp]
    lib.cts_last_error.restype = C.c_char_p
    lib.cts_ts_patch_count.argtypes = [vp, vp, i, i, i, i, i, vp, vp, vp, vp, vp]
    lib.cts_ts_patchify.argtypes = [vp, vp, i, i, i, i, i, i, vp, i, i, vp, vp, vp, i, vp, i, vp]
    lib.cts_gemm.argtypes = [vp, C.POINTER(GemmArgs), vp]
    lib.cts_gemm_suggest_split.argtypes = [vp, ll, ll, ll, i]
    lib.cts_reduce_bias_act.argtypes = [vp, vp, i, ll, ll, vp, i, vp, ll, vp, i, vp]
    lib.cts_reduce_residual_rmsnorm.argtypes = [vp, vp, i, vp, vp, vp, f, vp, ll, ll, i, vp]
    lib.cts_reduce_swiglu.argtypes = [vp, vp, i, ll, ll, vp, i, i, vp]
    lib.cts_qkv_rope_cache.argtypes = [vp, vp, i, i, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, ll, i, i, i, i, vp, vp, f, i, vp]
    lib.cts_embed_gather.argtypes = [vp, vp, vp, vp, ll, ll, ll, i, vp]
    lib.cts_attn_prefill.argtypes = [vp, vp, vp, vp, vp, i, i, ll, i, i, i, f, vp, i, vp]
    lib.cts_attn_decode_workspace_floats.argtypes = [i, i, i, i]
    lib.cts_attn_decode_workspace_floats.restype = ll
    lib.cts_attn_decode.argtypes = [vp, vp, vp, vp, i, vp, i, vp, i, i, i, i, i, f, i, vp, vp, i, vp]
    lib.cts_greedy_advance.argtypes = [vp, vp, ll, i, vp, i, vp, vp, vp, vp, vp, vp, i, i, i, vp]
    lib.cts_ipc_alloc.argtypes = [vp, ll, C.POINTER(vp), C.c_char_p]
    lib.cts_ipc_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    lib.cts_ipc_close.argtypes = [vp, vp]
    lib.cts_ipc_free.argtypes = [vp, vp]
    lib.cts_peer_allreduce_residual_rmsnorm.argtypes = [vp, vp, i, vp, vp, vp, i, i, i, vp, vp, vp, f, vp, ll, ll, i, vp]
    lib.cts_peer_ll_region_bytes.argtypes = [i, i, ll]
    lib.cts_peer_ll_region_bytes.restype = ll
    lib.cts_peer_allreduce_ll.argtypes = [vp, vp, i, vp, ll, vp, i, i, i, vp, vp, vp, f, vp, ll, ll, i, vp]
    lib.cts_peer_allreduce_ll.restype = i
    lib.cts_trace_enable.argtypes = [vp, vp]
    lib.cts_gemm_w4.argtypes = [vp, C.POINTER(GemmW4Args), vp]
    lib.cts_gemm_w4_suggest_split.argtypes = [vp, ll, ll]
    lib.cts_gemm_w4_mma.argtypes = [vp, C.POINTER(GemmW4fArgs), vp]
    lib.cts_gemm_w4_mma_suggest_split.argtypes = [vp, ll, ll, ll]
    lib.cts_gemm_w4_prefill.argtypes = [vp, C.POINTER(GemmW4pArgs), vp]
    lib.cts_rep_penalty_mark.argtypes = [vp, vp, vp, i, vp, i, ll, vp]
    lib.cts_rep_penalty_apply.argtypes = [vp, vp, ll, ll, i, vp, i, f, i, vp]
    lib.cts_ts_encode_fused_ok.argtypes = [C.POINTER(TsEncodeArgs)]
    lib.cts_ts_encode_fused.argtypes = [vp, C.POINTER(TsEncodeArgs), vp]
    lib.cts_decode_chain.argtypes = [vp, C.POINTER(ChainArgs), vp]
    lib.cts_decode_chain.restype = i
    lib.cts_peer_greedy_advance.argtypes = [vp, vp, ll, i, i, i, vp, vp, vp, i, vp, i, vp, vp, vp, vp, vp, vp, i, i, i, vp]
    lib.cts_peer_greedy_advance.restype = i
    lib.cts_gemm_decode_fused.argtypes = [vp, C.POINTER(FusedGemmArgs), vp]
    lib.cts_gemm_decode_fused.restype = i
    lib.cts_ts_encode.argtypes = [vp, C.POINTER(TsEncodeArgs), vp]
    lib.cts_ts_encode.restype = i
    lib.cts_rmsnorm.argtypes = [vp, vp, vp, f, vp, ll, ll, i, vp]
    lib.cts_lm_head.argtypes = [vp, vp, vp, vp, ll, ll, ll, i, vp]
    lib.cts_decoder_step_ws_floats.argtypes = [C.POINTER(DecoderStepArgs)]
    lib.cts_decoder_step_ws_floats.restype = ll
    lib.cts_decoder_step.argtypes = [vp, C.POINTER(DecoderStepArgs), vp]
    for name in ("cts_rmsnorm", "cts_lm_head", "cts_decoder_step"):
        getattr(lib, name).restype = i
    lib.cts_sample_advance.argtypes = [vp, vp, ll, i, f, i, f, C.c_ulonglong, vp, i, vp, vp, vp, vp, vp, vp, i, i, i, vp]
    lib.cts_sample_advance.restype = i
    # ---- A9: LoRA fine-tune step
    lib.cts_attn_prefill_lse.argtypes = [vp, vp, vp, vp, vp, i, i, ll, i, i, i, f, vp, vp, i, vp]
    lib.cts_attn_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i, i, ll, i, i, i, f, vp, vp, vp, vp, i, vp]
    lib.cts_swiglu.argtypes = [vp, vp, ll, ll, i, vp, i, vp]
    lib.cts_swiglu_bwd.argtypes = [vp, vp, vp, ll, ll, i, vp, i, vp]
    lib.cts_rmsnorm_bwd.argtypes = [vp, vp, vp, vp, f, vp, vp, ll, ll, i, vp]
    lib.cts_qkv_rope_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, f, vp, ll, i, i, i, i, vp]
    lib.cts_ce_loss_grad.argtypes = [vp, vp, ll, vp, ll, ll, f, vp, vp, i, i, vp]
    lib.cts_gather_rows.argtypes = [vp, vp, vp, ll, ll, vp, i, vp]
    lib.cts_lora_wgrad.argtypes = [vp, vp, ll, ll, i, ll, vp, ll, ll, i, ll, f, vp, ll, ll, i, vp]
    lib.cts_adamw.argtypes = [vp, vp, vp, vp, vp, ll, f, f, f, f, f, i, vp, vp]
    lib.cts_grad_norm_ws_floats.argtypes = []
    lib.cts_grad_norm_ws_floats.restype = ll
    lib.cts_grad_norm_clip.argtypes = [vp, vp, ll, f, vp, vp, vp]
    lib.cts_lora_pack.argtypes = [vp, vp, vp, i, ll, vp, i, vp]
    for name in ("cts_attn_prefill_lse", "cts_attn_bwd", "cts_swiglu", "cts_swiglu_bwd", "cts_rmsnorm_bwd", "cts_qkv_rope_bwd",
                 "cts_ce_loss_grad", "cts_gather_rows", "cts_lora_wgrad", "cts_adamw", "cts_grad_norm_clip", "cts_lora_pack"):
        getattr(lib, name).restype = i
    for name in ("cts_ipc_alloc", "cts_ipc_open", "cts_ipc_close", "cts_ipc_free", "cts_peer_allreduce_residual_rmsnorm"):
        getattr(lib, name).restype = i
    for name in ("cts_ts_patch_count", "cts_ts_patchify", "cts_gemm", "cts_gemm_suggest_split", "cts_reduce_bias_act",
                 "cts_reduce_residual_rmsnorm", "cts_reduce_swiglu", "cts_qkv_rope_cache", "cts_embed_gather",
                 "cts_attn_prefill", "cts_attn_decode", "cts_greedy_advance", "cts_ctx_create"):
        getattr(lib, name).restype = i
    _lib = lib
    return lib


def dtype_code(dt):
    if dt == torch.bfloat16:
        return BF16
    if dt == torch.float16:
        return F16
    raise CtsError(f"unsupported model dtype {dt}: the sm_100a kernels compute in bf16 or fp16 with fp32 accumulate")


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Context:
    """One per (process, device).  Raises if the GPU is not sm_100 -- there is nothing else to run on."""

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise CtsError("no CUDA device visible: chatts_b200 runs on B200 (sm_100a) only, with no CPU fallback")
        self.lib = load_library()
        self.device = torch.cuda.current_device() if device is None else torch.device(device).index or 0
        h = C.c_void_p()
        rc = self.lib.cts_ctx_create(self.device, C.byref(h))
        if rc != OK or not h:
            raise CtsError(f"cts_ctx_create(device={self.device}) failed with {rc} (needs an sm_100 device)")
        self.h = h
        self.arch = self.lib.cts_arch().decode()
        self.launches = 0          # kernels launched through this ctx (bench.py's gpu_launches evidence)
        # CTS_DEBUG_SYNC=1: synchronise after every entry point and name the one whose kernel faulted (asynchronous CUDA errors
        # otherwise surface at some later, unrelated call).  Debugging aid only -- never on in a measurement.
        self._debug_sync = os.environ.get("CTS_DEBUG_SYNC", "0") == "1"

    def close(self):
        if getattr(self, "h", None):
            self.lib.cts_ctx_destroy(self.h)
            self.h = None

    def _chk(self, rc, n_kernels=1):
        self.launches += n_kernels
        if rc != OK:
            raise CtsError(f"chatts_b200 error {rc}: {self.lib.cts_last_error(self.h).decode()}")
        if self._debug_sync and not torch.cuda.is_current_stream_capturing():
            try:
                torch.cuda.synchronize()
            except Exception as e:
                import sys
                raise CtsError(f"kernel fault inside Context.{sys._getframe(1).f_code.co_name}: {e}") from e

    # ------------------------------------------------------------------ device-side timeline (debug aid, csrc/trace.cuh)
    def trace_begin(self, capacity=1 << 20):
        buf = torch.zeros(2 + 2 * capacity, dtype=torch.int64, device=f"cuda:{self.device}")
        buf[1] = capacity
        torch.cuda.synchronize()
        rc = self.lib.cts_trace_enable(self.h, _p(buf))
        if rc != OK:
            raise CtsError(self.lib.cts_last_error(self.h).decode())
        self._trace = buf
        return buf

    def trace_end(self):
        """-> int64 array [n, 2] of {tag, globaltimer ns} records; tracing is switched off."""
        torch.cuda.synchronize()
        self.lib.cts_trace_enable(self.h, None)
        buf, self._trace = self._trace, None
        n = min(int(buf[0]), int(buf[1]))
        return buf[2: 2 + 2 * n].view(n, 2).cpu().numpy()

    # ------------------------------------------------------------------ TS front end
    def ts_patch_count(self, x, num_features, patch_size):
        n = x.shape[0]
        row_len = x.numel() // max(n, 1)
        dev = x.device
        valid = torch.empty(n, dtype=torch.int32, device=dev)
        cnt = torch.empty(n, dtype=torch.int32, device=dev)
        off = torch.empty(n + 1, dtype=torch.int32, device=dev)
        mx = torch.empty(1, dtype=torch.int32, device=dev)
        self._chk(self.lib.cts_ts_patch_count(self.h, _p(x), dtype_code(x.dtype), n, row_len, num_features, patch_size,
                                              _p(valid), _p(cnt), _p(off), _p(mx), _stream()), 2)
        return valid, cnt, off, mx

    def ts_patchify(self, x, num_features, patch_size, mode, pos_table, emb_dim, max_seq_len, valid, off, mx,
                    max_patches, rows_out):
        n = x.shape[0]
        row_len = x.numel() // max(n, 1)
        self._chk(self.lib.cts_ts_patchify(self.h, _p(x), dtype_code(x.dtype), n, row_len, num_features, patch_size, mode,
                                           _p(pos_table), emb_dim, max_seq_len, _p(valid), _p(off), _p(mx), max_patches,
                                           _p(rows_out), rows_out.shape[1], _stream()))

    # ------------------------------------------------------------------ GEMM
    def suggest_split(self, n, k, t, dual=False):
        return int(self.lib.cts_gemm_suggest_split(self.h, n, k, t, int(dual)))

    def gemm(self, x, w, out, *, w2=None, bias=None, residual=None, row_map=None, epilogue=EPI_NONE, split_k=1, t=None,
             splitk_ws=None, tile_counters=None, next_w=None, next_split=1, next_bytes=0):
        """out[T,N] (or fp32 partial [S,T,N]) = x[T,K] @ w[N,K]^T with the fused epilogue.
        next_w / next_split / next_bytes: the weight the next GEMM of the chain streams (L2 prefetch hint, decode-sized t)."""
        a = GemmArgs()
        if next_w is not None and next_bytes > 0:
            a.next_w, a.next_n, a.next_k, a.next_ld = next_w.data_ptr(), next_w.shape[0], next_w.shape[1], next_w.stride(0)
            a.next_split, a.next_prefetch_bytes = int(next_split), int(next_bytes)
        a.w, a.w2, a.x = w.data_ptr(), (w2.data_ptr() if w2 is not None else None), x.data_ptr()
        a.bias = bias.data_ptr() if bias is not None else None
        a.residual = residual.data_ptr() if residual is not None else None
        a.out = out.data_ptr()
        a.row_map = row_map.data_ptr() if row_map is not None else None
        a.n, a.k = w.shape[0], w.shape[1]
        a.t = x.shape[0] if t is None else t
        a.w_ld, a.x_ld = w.stride(0), x.stride(0)
        a.out_ld = out.stride(-2) if epilogue not in (EPI_PARTIAL_F32, EPI_SPLITK_F32) else a.n
        a.splitk_ws = splitk_ws.data_ptr() if splitk_ws is not None else None
        a.tile_counters = tile_counters.data_ptr() if tile_counters is not None else None
        a.dtype, a.epilogue, a.split_k = dtype_code(x.dtype), epilogue, split_k
        self._chk(self.lib.cts_gemm(self.h, C.byref(a), _stream()))

    def gemm_w4(self, x, qw, scales, zeros, group_size, out, split_k, t=None):
        """fp32 split-K partials [S, T, N] of x[T, K] @ W^T with W = scales * (codes - zeros) dequantised in the operand path
        (cts_gemm_w4; decode-sized T).  qw uint8 [N, K/2], scales [N, K/g] (x's dtype), zeros uint8 [N, K/g]."""
        a = GemmW4Args()
        a.qw, a.scales, a.zeros, a.x, a.out = qw.data_ptr(), scales.data_ptr(), zeros.data_ptr(), x.data_ptr(), out.data_ptr()
        a.n, a.k = qw.shape[0], qw.shape[1] * 2
        a.t = x.shape[0] if t is None else t
        a.x_ld, a.group_size, a.split_k, a.dtype = x.stride(0), int(group_size), int(split_k), dtype_code(x.dtype)
        self._chk(self.lib.cts_gemm_w4(self.h, C.byref(a), _stream()))

    def gemm_w4_suggest_split(self, n, k):
        return int(self.lib.cts_gemm_w4_suggest_split(self.h, n, k))

    def gemm_w4_mma(self, x, qwf, szp, n, group_size, out, split_k, t=None):
        """The same partials with the weight operand dequantised in registers (cts_gemm_w4_mma).  qwf uint8 [ceil(N/256) * K/64 * 8192]
        fragment-major codes, szp int32 [ceil(N/256), K/g, 256] (weights.py:repack_w4_mma); n = the true number of features."""
        a = GemmW4fArgs()
        a.qw, a.szp, a.x, a.out = qwf.data_ptr(), szp.data_ptr(), x.data_ptr(), out.data_ptr()
        a.n, a.k = int(n), szp.shape[1] * int(group_size)
        a.t = x.shape[0] if t is None else t
        a.x_ld, a.group_size, a.split_k, a.dtype = x.stride(0), int(group_size), int(split_k), dtype_code(x.dtype)
        self._chk(self.lib.cts_gemm_w4_mma(self.h, C.byref(a), _stream()))

    def gemm_w4_mma_suggest_split(self, n, k, t=1):
        return int(self.lib.cts_gemm_w4_mma_suggest_split(self.h, n, k, t))

    def gemm_w4_prefill(self, x, qwf, szp, n, group_size, out, *, bias=None, residual=None, epilogue=EPI_NONE, split_k=1, t=None):
        """cts_gemm's epilogues (NONE / RESIDUAL / SWIGLU_IL / PARTIAL_F32) over the fragment-major 4-bit weight of gemm_w4_mma
        (cts_gemm_w4_prefill: persistent tcgen05 GEMM, any t): bit-identical to gemm() on weights.py:dequantize_w4 of the same codes."""
        a = GemmW4pArgs()
        a.qw, a.szp, a.x, a.out = qwf.data_ptr(), szp.data_ptr(), x.data_ptr(), out.data_ptr()
        a.bias = bias.data_ptr() if bias is not None else None
        a.residual = residual.data_ptr() if residual is not None else None
        a.n, a.k = int(n), szp.shape[1] * int(group_size)
        a.t = x.shape[0] if t is None else t
        a.x_ld = x.stride(0)
        a.out_ld = out.stride(-2) if epilogue != EPI_PARTIAL_F32 else a.n
        a.group_size, a.split_k, a.dtype, a.epilogue = int(group_size), int(split_k), dtype_code(x.dtype), int(epilogue)
        self._chk(self.lib.cts_gemm_w4_prefill(self.h, C.byref(a), _stream()))

    # ------------------------------------------------------------------ fused split-K tails
    def reduce_bias_act(self, partial, split_k, t, n, bias, act, out, row_map=None):
        self._chk(self.lib.cts_reduce_bias_act(self.h, _p(partial), split_k, t, n, _p(bias), act, _p(out), out.stride(0),
                                               _p(row_map), dtype_code(out.dtype), _stream()))

    def reduce_residual_rmsnorm(self, partial, split_k, resid_in, resid_out, norm_w, eps, norm_out, t=None):
        t = resid_in.shape[0] if t is None else t
        self._chk(self.lib.cts_reduce_residual_rmsnorm(self.h, _p(partial), split_k, _p(resid_in), _p(resid_out), _p(norm_w),
                                                       float(eps), _p(norm_out), t, resid_in.shape[-1],
                                                       dtype_code(resid_in.dtype), _stream()))

    def reduce_swiglu(self, partial, split_k, t, inter, out, interleaved=False):
        self._chk(self.lib.cts_reduce_swiglu(self.h, _p(partial), split_k, t, inter, _p(out), int(interleaved),
                                             dtype_code(out.dtype), _stream()))

    def qkv_rope_cache(self, src, src_is_partial, split_k, bias, positions, cos, sin, slot_map, q_out, k_cache, v_cache,
                       k_out, v_out, t, nh, nkv, head_dim, page_size, q_norm_w=None, k_norm_w=None, norm_eps=1e-6):
        self._chk(self.lib.cts_qkv_rope_cache(self.h, _p(src), int(src_is_partial), split_k, _p(bias), _p(positions), _p(cos),
                                              _p(sin), _p(slot_map), _p(q_out), _p(k_cache), _p(v_cache), _p(k_out), _p(v_out),
                                              t, nh, nkv, head_dim, page_size, _p(q_norm_w), _p(k_norm_w), float(norm_eps),
                                              dtype_code(q_out.dtype), _stream()))

    def embed_gather(self, table, ids, out, t=None):
        t = ids.shape[0] if t is None else t
        self._chk(self.lib.cts_embed_gather(self.h, _p(table), _p(ids), _p(out), t, table.shape[1], table.shape[0],
                                            dtype_code(table.dtype), _stream()))

    # ------------------------------------------------------------------ attention
    def attn_prefill(self, q, k, v, cu_seqlens, batch, max_seqlen, nh, nkv, head_dim, scale, out):
        self._chk(self.lib.cts_attn_prefill(self.h, _p(q), _p(k), _p(v), _p(cu_seqlens), batch, max_seqlen, q.shape[0], nh, nkv,
                                            head_dim, float(scale), _p(out), dtype_code(q.dtype), _stream()))

    def attn_decode_workspace_floats(self, batch, nh, head_dim, num_splits):
        return int(self.lib.cts_attn_decode_workspace_floats(batch, nh, head_dim, num_splits))

    def attn_decode(self, q, k_cache, v_cache, page_table, seq_lens, batch, nh, nkv, head_dim, page_size, scale, num_splits,
                    workspace, out):
        self._chk(self.lib.cts_attn_decode(self.h, _p(q), _p(k_cache), _p(v_cache), k_cache.shape[0], _p(page_table),
                                           page_table.shape[1], _p(seq_lens), batch, nh, nkv, head_dim, page_size, float(scale),
                                           num_splits, _p(workspace), _p(out), dtype_code(q.dtype), _stream()))

    def greedy_advance(self, logits, batch, out_tokens, step_ptr, cur_ids, positions, seq_lens, slot_map, page_table,
                       page_size):
        self._chk(self.lib.cts_greedy_advance(self.h, _p(logits), logits.shape[-1], batch, _p(out_tokens),
                                              out_tokens.stride(0) if out_tokens is not None else 0, _p(step_ptr), _p(cur_ids),
                                              _p(positions), _p(seq_lens), _p(slot_map), _p(page_table),
                                              page_table.shape[1] if page_table is not None else 0, page_size,
                                              dtype_code(logits.dtype), _stream()))

    def gemm_decode_fused(self, x, w, mode, split_k, t, *, bias=None, h=None, act=None, positions=None, cos=None, sin=None, slot_map=None,
                          q_out=None, k_cache=None, v_cache=None, q_norm=None, k_norm=None, eps=1e-6, nh=0, nkv=0, head_dim=0,
                          page_size=0, norm_h=None, norm_w=None, ssq_in=None, norm_eps=1e-6, ssq_out=None, peer=None):
        """Cluster-reduced decode GEMM with the projection's tail fused in (cts_gemm_decode_fused); t <= 32, split_k <= 8.
        norm_h / norm_w / ssq_in: the token operand is RMSNorm(norm_h) produced inside the kernel (x may be None);
        ssq_out (RESIDUAL): per-tile sums of squares of the updated h for the next projection's fused RMSNorm;
        peer (RESIDUAL, row-parallel under TP): the all-reduce over peer memory happens inside the kernel."""
        a = FusedGemmArgs()
        dp = lambda v: None if v is None else v.data_ptr()
        a.w, a.x, a.n, a.k, a.t = w.data_ptr(), dp(x), w.shape[0], w.shape[1], t
        a.norm_h, a.norm_w, a.ssq_in, a.ssq_out = dp(norm_h), dp(norm_w), dp(ssq_in), dp(ssq_out)
        a.ssq_tiles, a.norm_eps = (ssq_in.shape[-1] if ssq_in is not None else 0), float(norm_eps)
        a.dtype, a.mode, a.split_k = dtype_code(w.dtype), int(mode), int(split_k)
        a.bias, a.h, a.act = dp(bias), dp(h), dp(act)
        a.positions, a.cos_tab, a.sin_tab, a.slot_map = dp(positions), dp(cos), dp(sin), dp(slot_map)
        a.q_out, a.k_cache, a.v_cache, a.q_norm, a.k_norm = dp(q_out), dp(k_cache), dp(v_cache), dp(q_norm), dp(k_norm)
        a.eps, a.nh, a.nkv, a.head_dim, a.page_size = float(eps), nh, nkv, head_dim, page_size
        if peer is not None:            # (regions, region_bytes, state, rank, world, max_tokens): row-parallel projection under TP
            a.peer_regions, a.peer_region_bytes, a.peer_state = peer[0].data_ptr(), int(peer[1]), peer[2].data_ptr()
            a.peer_rank, a.peer_world, a.peer_max_tokens = int(peer[3]), int(peer[4]), int(peer[5])
        self._chk(self.lib.cts_gemm_decode_fused(self.h, C.byref(a), _stream()))

    def ts_encode(self, x, num_features, patch_size, mode, pos_table, emb_dim, max_seq_len, weights, biases, total_rows, out, row_map=None):
        """cts_ts_encode: counts + patchify + the whole MLP from one C call.  ``total_rows`` is the host-known sum of the patch
        counts.  Returns (valid_len, patch_cnt, row_offset) device tensors."""
        n = x.shape[0]
        xx = x.reshape(n, -1).contiguous()
        dev, dt = xx.device, xx.dtype
        hidden, in0 = weights[0].shape[0], weights[0].shape[1]
        valid = torch.empty(n, dtype=torch.int32, device=dev)
        cnt = torch.empty(n, dtype=torch.int32, device=dev)
        off = torch.empty(n + 1, dtype=torch.int32, device=dev)
        mx = torch.empty(1, dtype=torch.int32, device=dev)
        rows = torch.empty(max(total_rows, 1), in0, device=dev, dtype=dt)
        act = [torch.empty(max(total_rows, 1), hidden, device=dev, dtype=dt) for _ in range(2)]
        ws = torch.empty(16 * max(total_rows, 1) * hidden, device=dev, dtype=torch.float32)
        a = TsEncodeArgs()
        a.x, a.dtype, a.n_series, a.row_len = xx.data_ptr(), dtype_code(dt), n, xx.shape[1]
        a.num_features, a.patch_size, a.mode = num_features, patch_size, mode
        a.pos_table = pos_table.data_ptr() if pos_table is not None else None
        a.emb_dim, a.max_seq_len, a.num_layers, a.hidden, a.in0 = emb_dim, max_seq_len, len(weights), hidden, in0
        wt = (C.c_void_p * len(weights))(*[w.data_ptr() for w in weights])
        bt = (C.c_void_p * len(biases))(*[b.data_ptr() for b in biases])
        a.weights, a.biases = wt, bt
        a.valid_len, a.patch_cnt, a.row_offset, a.max_valid = valid.data_ptr(), cnt.data_ptr(), off.data_ptr(), mx.data_ptr()
        a.total_rows = total_rows
        a.rows_ws, a.splitk_ws, a.splitk_floats = rows.data_ptr(), ws.data_ptr(), ws.numel()
        a.act_ws[0], a.act_ws[1] = act[0].data_ptr(), act[1].data_ptr()
        a.out, a.out_ld = out.data_ptr(), out.stride(0)
        a.row_map = row_map.data_ptr() if row_map is not None else None
        self._chk(self.lib.cts_ts_encode(self.h, C.byref(a), _stream()), 3 + 2 * len(weights))
        return valid, cnt, off

    def ts_mlp_fused(self, x, num_features, patch_size, mode, pos_table, emb_dim, max_seq_len, weights, biases, valid, off, mx,
                     total_rows, out, row_map=None):
        """cts_ts_encode_fused: patchify + the whole MLP + the row scatter in ONE launch (<= 256 patch rows; the count stage has run:
        ``valid`` / ``off`` / ``mx`` are its outputs).  Returns False when the shape is outside the fused kernel's range."""
        n = x.shape[0]
        xx = x.reshape(n, -1)
        dev, dt = xx.device, xx.dtype
        hidden, in0 = weights[0].shape[0], weights[0].shape[1]
        a = TsEncodeArgs()
        a.x, a.dtype, a.n_series, a.row_len = xx.data_ptr(), dtype_code(dt), n, xx.shape[1]
        a.num_features, a.patch_size, a.mode = num_features, patch_size, mode
        a.pos_table = pos_table.data_ptr() if pos_table is not None else None
        a.emb_dim, a.max_seq_len, a.num_layers, a.hidden, a.in0 = emb_dim, max_seq_len, len(weights), hidden, in0
        a.total_rows = total_rows
        if not self.lib.cts_ts_encode_fused_ok(C.byref(a)):
            return False
        key = (total_rows, in0, hidden, str(dt), str(dev))
        cache = self.__dict__.setdefault("_ts_fused_ws", {})
        ws = cache.get(key)
        if ws is None:                                  # persistent workspaces: stable addresses under CUDA-graph capture
            ws = (torch.empty(total_rows, in0, device=dev, dtype=dt), [torch.empty(total_rows, hidden, device=dev, dtype=dt) for _ in range(2)])
            cache[key] = ws
        rows, act = ws
        wt = (C.c_void_p * len(weights))(*[w.data_ptr() for w in weights])
        bt = (C.c_void_p * len(biases))(*[b.data_ptr() for b in biases])
        a.weights, a.biases = wt, bt
        a.valid_len, a.row_offset, a.max_valid = valid.data_ptr(), off.data_ptr(), mx.data_ptr()
        a.rows_ws = rows.data_ptr()
        a.act_ws[0], a.act_ws[1] = act[0].data_ptr(), act[1].data_ptr()
        a.out, a.out_ld = out.data_ptr(), out.stride(0)
        a.row_map = row_map.data_ptr() if row_map is not None else None
        self._chk(self.lib.cts_ts_encode_fused(self.h, C.byref(a), _stream()), 1)
        return True

    def rmsnorm(self, x, w, eps, out, t=None):
        t = x.shape[0] if t is None else t
        self._chk(self.lib.cts_rmsnorm(self.h, _p(x), _p(w), float(eps), _p(out), t, x.shape[-1], dtype_code(x.dtype), _stream()))

    def lm_head(self, hidden, w, logits, t=None):
        t = hidden.shape[0] if t is None else t
        self._chk(self.lib.cts_lm_head(self.h, _p(hidden), _p(w), _p(logits), t, w.shape[1], w.shape[0], dtype_code(hidden.dtype), _stream()))

    def decoder_step(self, *, layers, embed, final_norm, lm_head, cos, sin, hidden, inter, nh, nkv, head_dim, eps, page_size, batch,
                     splits, attn_splits, cur_ids, positions, seq_lens, slot_map, page_table, out_tokens, step_ptr, h, xn, q, ao, act,
                     logits, ws, attn_ws, sample=True):
        """One whole decode step enqueued by ONE C call (cts_decoder_step).  ``layers``: list of dicts of tensors (wqkv, bqkv,
        q_norm, k_norm, wo, wgu, wd, ln1, ln2, k_cache, v_cache); ``splits`` = (qkv, o, gu, d).  The ctypes layer table is
        cached per list object."""
        key = id(layers)
        cache = self.__dict__.setdefault("_layer_tables", {})
        if key not in cache:
            arr = (LayerWeights * len(layers))()
            for i2, lw in enumerate(layers):
                for f2, _ in LayerWeights._fields_:
                    t2 = lw.get(f2)
                    setattr(arr[i2], f2, None if t2 is None else t2.data_ptr())
            cache[key] = (arr, layers)                       # keep the list alive: the table holds raw pointers into it
        arr = cache[key][0]
        a = DecoderStepArgs()
        a.n_layers, a.hidden, a.inter, a.nh, a.nkv, a.head_dim = len(layers), hidden, inter, nh, nkv, head_dim
        a.vocab, a.vocab_rows = lm_head.shape[0], embed.shape[0]
        a.page_size, a.num_pages, a.max_pages = page_size, layers[0]["k_cache"].shape[0], page_table.shape[1]
        a.dtype, a.batch, a.sample, a.eps = dtype_code(h.dtype), batch, int(bool(sample)), float(eps)
        a.split_qkv, a.split_o, a.split_gu, a.split_d = (int(v) for v in splits)
        a.attn_splits = int(attn_splits)
        a.layers = arr
        dp = lambda x: None if x is None else x.data_ptr()
        a.embed, a.final_norm, a.lm_head, a.cos_tab, a.sin_tab = dp(embed), dp(final_norm), dp(lm_head), dp(cos), dp(sin)
        a.cur_ids, a.positions, a.seq_lens, a.slot_map, a.page_table = dp(cur_ids), dp(positions), dp(seq_lens), dp(slot_map), dp(page_table)
        a.out_tokens, a.out_ld, a.step_ptr = dp(out_tokens), (out_tokens.stride(0) if out_tokens is not None else 0), dp(step_ptr)
        a.h, a.xn, a.q, a.ao, a.act, a.logits = dp(h), dp(xn), dp(q), dp(ao), dp(act), dp(logits)
        a.ws, a.ws_floats, a.attn_ws = dp(ws), ws.numel(), dp(attn_ws)
        need = int(self.lib.cts_decoder_step_ws_floats(C.byref(a)))
        if ws.numel() < need:
            raise CtsError(f"decoder_step: split-K workspace holds {ws.numel()} floats, {need} needed")
        self._chk(self.lib.cts_decoder_step(self.h, C.byref(a), _stream()), 3 + 9 * len(layers) + int(bool(sample)))

    def sample_advance(self, logits, batch, temperature, top_k, top_p, seed, out_tokens, step_ptr, cur_ids, positions, seq_lens,
                       slot_map, page_table, page_size):
        self._chk(self.lib.cts_sample_advance(self.h, _p(logits), logits.shape[-1], batch, float(temperature), int(top_k or 0),
                                              float(top_p if top_p is not None else 1.0), int(seed) & 0xFFFFFFFFFFFFFFFF, _p(out_tokens),
                                              out_tokens.stride(0) if out_tokens is not None else 0, _p(step_ptr), _p(cur_ids),
                                              _p(positions), _p(seq_lens), _p(slot_map), _p(page_table),
                                              page_table.shape[1] if page_table is not None else 0, page_size,
                                              dtype_code(logits.dtype), _stream()))

    def rep_penalty_mark(self, tokens, rows, seen, vocab):
        """Set the bits of (row, token) pairs in seen [B, words]; rows None: pair i belongs to row i."""
        self._chk(self.lib.cts_rep_penalty_mark(self.h, _p(tokens), _p(rows), tokens.numel(), _p(seen), seen.shape[1], vocab, _stream()))

    def rep_penalty_apply(self, logits, batch, seen, penalty):
        self._chk(self.lib.cts_rep_penalty_apply(self.h, _p(logits), logits.shape[-1], logits.stride(0), batch, _p(seen), seen.shape[1],
                                                 float(penalty), dtype_code(logits.dtype), _stream()))

    # ------------------------------------------------------------------ A9: LoRA fine-tune step
    def attn_prefill_lse(self, q, k, v, cu_seqlens, batch, max_seqlen, nh, nkv, head_dim, scale, out, lse):
        self._chk(self.lib.cts_attn_prefill_lse(self.h, _p(q), _p(k), _p(v), _p(cu_seqlens), batch, max_seqlen, q.shape[0], nh, nkv,
                                                head_dim, float(scale), _p(out), _p(lse), dtype_code(q.dtype), _stream()))

    def attn_bwd(self, q, k, v, out, dout, lse, cu_seqlens, batch, max_seqlen, nh, nkv, head_dim, scale, delta_ws, dq, dk, dv):
        self._chk(self.lib.cts_attn_bwd(self.h, _p(q), _p(k), _p(v), _p(out), _p(dout), _p(lse), _p(cu_seqlens), batch, max_seqlen,
                                        q.shape[0], nh, nkv, head_dim, float(scale), _p(delta_ws), _p(dq), _p(dk), _p(dv),
                                        dtype_code(q.dtype), _stream()), 3)

    def swiglu(self, gu, t, inter, out, interleaved=True):
        self._chk(self.lib.cts_swiglu(self.h, _p(gu), t, inter, int(interleaved), _p(out), dtype_code(gu.dtype), _stream()))

    def swiglu_bwd(self, gu, dact, t, inter, dgu, interleaved=True):
        self._chk(self.lib.cts_swiglu_bwd(self.h, _p(gu), _p(dact), t, inter, int(interleaved), _p(dgu), dtype_code(gu.dtype),
                                          _stream()))

    def rmsnorm_bwd(self, dy, x, w, eps, dres_in, dx_out, t=None):
        t = x.shape[0] if t is None else t
        self._chk(self.lib.cts_rmsnorm_bwd(self.h, _p(dy), _p(x), _p(w), float(eps), _p(dres_in), _p(dx_out), t, x.shape[-1],
                                           dtype_code(x.dtype), _stream()))

    def qkv_rope_bwd(self, dq, dk, dv, qkv, positions, cos, sin, q_norm_w, k_norm_w, norm_eps, dqkv, t, nh, nkv, head_dim):
        self._chk(self.lib.cts_qkv_rope_bwd(self.h, _p(dq), _p(dk), _p(dv), _p(qkv), _p(positions), _p(cos), _p(sin), _p(q_norm_w),
                                            _p(k_norm_w), float(norm_eps), _p(dqkv), t, nh, nkv, head_dim, dtype_code(dq.dtype),
                                            _stream()))

    def ce_loss_grad(self, logits, targets, n_rows, grad_scale, row_loss, loss_out, accumulate=False):
        self._chk(self.lib.cts_ce_loss_grad(self.h, _p(logits), logits.stride(0), _p(targets), n_rows, logits.shape[1],
                                            float(grad_scale), _p(row_loss), _p(loss_out), int(accumulate),
                                            dtype_code(logits.dtype), _stream()), 2)

    def gather_rows(self, src, idx, n_out, dst):
        self._chk(self.lib.cts_gather_rows(self.h, _p(src), _p(idx), n_out, src.shape[-1], _p(dst), dtype_code(src.dtype), _stream()))

    def lora_wgrad(self, p, p_col0, p_il, m, q, q_col0, r, t, scale, out, so_m, so_r):
        """out[i*so_m + j*so_r] += scale * sum_t p[t, col(i)] * q[t, q_col0 + j]   (out: fp32 view into the gradient arena)"""
        self._chk(self.lib.cts_lora_wgrad(self.h, _p(p), p.stride(0), p_col0, int(p_il), m, _p(q), q.stride(0), q_col0, r, t,
                                          float(scale), _p(out), so_m, so_r, dtype_code(p.dtype), _stream()))

    def adamw(self, p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=None):
        self._chk(self.lib.cts_adamw(self.h, _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2), float(eps),
                                     float(weight_decay), int(step), _p(grad_scale), _stream()))

    def grad_norm_ws_floats(self):
        return int(self.lib.cts_grad_norm_ws_floats())

    def grad_norm_clip(self, g, max_norm, ws, out):
        self._chk(self.lib.cts_grad_norm_clip(self.h, _p(g), g.numel(), float(max_norm), _p(ws), _p(out), _stream()), 2)

    def lora_pack(self, master, desc, n_desc, max_elems, work):
        self._chk(self.lib.cts_lora_pack(self.h, _p(master), _p(desc), n_desc, max_elems, _p(work), dtype_code(work.dtype), _stream()))

    # ------------------------------------------------------------------ tensor parallel (peer memory)
    def ipc_alloc(self, nbytes):
        ptr = C.c_void_p()
        handle = C.create_string_buffer(64)
        self._chk(self.lib.cts_ipc_alloc(self.h, nbytes, C.byref(ptr), handle), 0)
        return ptr.value, handle.raw

    def ipc_open(self, handle):
        ptr = C.c_void_p()
        self._chk(self.lib.cts_ipc_open(self.h, handle, C.byref(ptr)), 0)
        return ptr.value

    def peer_allreduce_residual_rmsnorm(self, local_partial, split_k, peer_rows, peer_flags, state, rank, world, max_tokens, resid_in,
                                        resid_out, norm_w, eps, norm_out, t):
        self._chk(self.lib.cts_peer_allreduce_residual_rmsnorm(self.h, _p(local_partial), split_k, _p(peer_rows), _p(peer_flags), _p(state),
                                                               rank, world, max_tokens, _p(resid_in), _p(resid_out), _p(norm_w),
                                                               float(eps), _p(norm_out), t, resid_in.shape[-1],
                                                               dtype_code(resid_in.dtype), _stream()))

    def peer_ll_region_bytes(self, world, max_tokens, h):
        return int(self.lib.cts_peer_ll_region_bytes(world, max_tokens, h))

    def peer_allreduce_ll(self, local_partial, split_k, peer_regions, region_bytes, state, rank, world, max_tokens, resid_in, resid_out,
                          norm_w, eps, norm_out, t):
        self._chk(self.lib.cts_peer_allreduce_ll(self.h, _p(local_partial), split_k, _p(peer_regions), region_bytes, _p(state), rank, world,
                                                 max_tokens, _p(resid_in), _p(resid_out), _p(norm_w), float(eps), _p(norm_out), t,
                                                 resid_in.shape[-1], dtype_code(resid_in.dtype), _stream()))

    def decode_chain(self, *, t, hidden, inter, nh, nkv, head_dim, phases, splits, h, xn, act, ws, ssq, sync, eps, dtype,
                     norm5_has_partial=1, wo=None, wgu=None, wd=None, wqkv=None, ao=None, ln_post=None, ln_next=None, bqkv=None,
                     q_norm_w=None, k_norm_w=None, positions=None, cos=None, sin=None, slot_map=None, q_out=None, k_cache=None,
                     v_cache=None, page_size=0):
        """One persistent kernel for the phases [phases[0], phases[1]) of a decode layer chain (include/chatts_b200.h)."""
        a = ChainArgs()
        a.t, a.hidden, a.inter, a.nh, a.nkv, a.head_dim = t, hidden, inter, nh, nkv, head_dim
        a.phase_begin, a.phase_end, a.norm5_has_partial, a.dtype = phases[0], phases[1], int(norm5_has_partial), dtype_code(dtype)
        for i2, v in enumerate(splits):
            a.split[i2] = int(v)
        dp = lambda x: None if x is None else x.data_ptr()
        a.wo, a.wgu, a.wd, a.wqkv, a.ao = dp(wo), dp(wgu), dp(wd), dp(wqkv), dp(ao)
        a.h, a.xn, a.act, a.ln_post, a.ln_next, a.eps = dp(h), dp(xn), dp(act), dp(ln_post), dp(ln_next), float(eps)
        a.bqkv, a.q_norm_w, a.k_norm_w = dp(bqkv), dp(q_norm_w), dp(k_norm_w)
        a.positions, a.cos_tab, a.sin_tab, a.slot_map = dp(positions), dp(cos), dp(sin), dp(slot_map)
        a.q_out, a.k_cache, a.v_cache, a.page_size = dp(q_out), dp(k_cache), dp(v_cache), int(page_size)
        a.ws, a.ssq, a.sync = dp(ws), dp(ssq), dp(sync)
        self._chk(self.lib.cts_decode_chain(self.h, C.byref(a), _stream()))

    def peer_greedy_advance(self, logits, batch, rank, world, peer_cand, peer_flags, state, max_batch, out_tokens, step_ptr, cur_ids,
                            positions, seq_lens, slot_map, page_table, page_size):
        self._chk(self.lib.cts_peer_greedy_advance(self.h, _p(logits), logits.shape[-1], batch, rank, world, _p(peer_cand), _p(peer_flags),
                                                   _p(state), max_batch, _p(out_tokens), out_tokens.stride(0), _p(step_ptr), _p(cur_ids),
                                                   _p(positions), _p(seq_lens), _p(slot_map), _p(page_table), page_table.shape[1],
                                                   page_size, dtype_code(logits.dtype), _stream()))


_ctx_cache = {}


def get_context(device=None):
    dev = torch.cuda.current_device() if device is None else (torch.device(device).index or 0)
    if dev not in _ctx_cache:
        with torch.cuda.device(dev):
            _ctx_cache[dev] = Context(dev)
    return _ctx_cache[dev]
