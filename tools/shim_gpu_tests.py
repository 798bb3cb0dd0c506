"""GPU tests executed on a machine WITHOUT a GPU through the "CUDA on CPU" shim (tests/cuda_on_cpu): `ctx()` returns a Context whose library
is the kernels' own source compiled by g++ -- CUDA threads as fibers, clusters as threads, and a functional emulation of mbarrier / TMA /
TMEM / tcgen05.mma that is calibrated by the GPU-validated GEMM kernels passing their own test file -- and `.cuda()` is the identity.
Unlike tools/dryrun_train_gpu_tests.py (which checks the TEST LOGIC against the torch double), this executes the KERNEL SOURCE.
TEST INFRASTRUCTURE ONLY.

    python tools/shim_gpu_tests.py [--quick] [pytest args]
"""
import functools
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pytest  # noqa: E402
import torch  # noqa: E402

for name in ("empty", "full", "zeros", "ones", "randn", "tensor", "empty_like", "zeros_like", "arange"):
    orig = getattr(torch, name)

    def mk(orig):
        @functools.wraps(orig)
        def f(*a, **k):
            if str(k.get("device", "")).startswith("cuda"):
                k.pop("device")
            return orig(*a, **k)
        return f
    setattr(torch, name, mk(orig))
if os.environ.get("CTS_SHIM_POISON") == "1":
    # "initcheck": every torch.empty / empty_like of a floating type comes back full of NaN, so a kernel that reads memory nobody wrote shows
    # up as NaN in a result that is compared with a reference
    for _n in ("empty", "empty_like"):
        _o = getattr(torch, _n)

        def _mk(_o):
            @functools.wraps(_o)
            def f(*a, **k):
                t = _o(*a, **k)
                if t.is_floating_point():
                    t.fill_(float("nan"))
                return t
            return f
        setattr(torch, _n, _mk(_o))
torch.Tensor.cuda = lambda self, *a, **k: self
_to = torch.Tensor.to


def _to_host(self, *a, **k):
    a = tuple(x for x in a if not (isinstance(x, (str, torch.device)) and "cuda" in str(x)))
    if "cuda" in str(k.get("device", "")):
        k.pop("device")
    k.pop("non_blocking", None)
    return _to(self, *a, **k) if (a or k) else self


torch.Tensor.to = _to_host
torch.cuda.synchronize = lambda *a, **k: None
torch.cuda.is_available = lambda: True
torch.cuda.current_device = lambda: 0
torch.cuda.is_current_stream_capturing = lambda: False

from tests.w4_prefill_support import shim_context_w4p  # noqa: E402
import tests.gpu_util as gu  # noqa: E402

_ctx = shim_context_w4p()                  # the standard shim library + csrc/gemm_w4_persistent.cu
from tests.cabi_double import TorchDouble as _TD  # noqa: E402
_dbl = _TD()
# HYBRID context for the whole-step tests: every entry point whose source is in the shim build runs that source; the others (tcgen05
# GEMMs, attention forward, the decode-side kernels) are answered by the torch double.  What this adds over the double-only dry run:
# train.py's argument plumbing (strides, interleaved layouts, arena offsets, packing descriptors) meets the REAL backward / loss /
# optimiser kernels.
_shim_native = []
for _name in dir(_TD):
    if _name.startswith("_") or not callable(getattr(_TD, _name)):
        continue
    try:
        getattr(_ctx.lib, "cts_" + _name)
        _shim_native.append(_name)
    except AttributeError:
        setattr(_ctx, _name, getattr(_dbl, _name))
from chatts_b200 import _cabi  # noqa: E402
_cabi.get_context = lambda device=None: _ctx
import chatts_b200.model as _mm  # noqa: E402
import chatts_b200.ts_encoder as _te  # noqa: E402
_mi, _ti = _mm.ChatTSForCausalLM.__init__, _te.TimeSeriesEmbedding.__init__


def _model_init(self, config, state_dict, device="cpu", **kw):
    kw["use_cuda_graph"] = False
    _mi(self, config, state_dict, device="cpu", **kw)


_mm.ChatTSForCausalLM.__init__ = _model_init
_mm.ChatTSForCausalLM.use_cuda_graph = property(lambda self: False, lambda self, v: None)      # no CUDA graphs on the host, whatever a test asks for
_te.TimeSeriesEmbedding.__init__ = lambda self, config, weights, device="cpu", **kw: _ti(self, config, weights, device="cpu", **kw)
torch.Tensor.pin_memory = lambda self: self
gu.ctx = lambda: _ctx
gu.record = lambda *a, **k: None

# the cases whose every entry point is part of the shim build
SELECT = {
    "test_gpu_zz_b_sampling.py": None,
    "test_gpu_zz_c_train.py": "adamw_and_clip or lora_pack or prefill_lse or test_attention_backward or train_step_matches_oracle or training_reduces_loss or (directional and False) or wgrad_tensor_core",
    "test_gpu_train_kernels.py": None,
    # the cluster-fused decode GEMMs against the two-launch path, BIT FOR BIT: both GEMM kernels run from source through the tcgen05 /
    # TMA / mbarrier emulation of the shim (same accumulation order), the reduce kernels of the two-launch path come from the double
    "test_gpu_zz_e_fused_decode.py": None,
    "test_gpu_gemm.py": None,                            # calibration of the emulation: the GPU-validated GEMM kernels themselves
    "test_gpu_elementwise.py": None,                     # calibration: split-K tails, RoPE / KV write, RMSNorm over a cluster (DSMEM), argmax + advance
    "test_gpu_ts_encoder.py": None,                      # calibration: the TS encoder against the reference-generated fixtures
    "test_gpu_zz_a_native_step.py": None,                # cts_decoder_step / cts_ts_encode: the C++ executors over the kernels above (pending on a B200)
    "test_gpu_model.py": "not full_size",                # calibration: the whole model (prefill, paged decode, generate, LoRA merge ...) from kernel source
    "test_gpu_attention.py": None,                       # calibration: tcgen05 prefill attention (MN-major V operand), HMMA prefill, TMA paged decode (ldmatrix / mma.sync)
    "test_gpu_zz_d_attn_bwd_tc5.py": None,               # tcgen05 attention backward (K-major and MN-major operands, TMEM-resident dQ / dK / dV)
    "test_gpu_w4.py": "not (27648 or 13824 or 7168)",    # both W4A16 kernels (tcgen05 operand path; registers + mma.sync over the persistent schedule), small shapes
    # aimed queries against the float64 reference: both prefill kernels on the varlen batch, the decode kernel over contexts up to 4097
    # (no split, the model's split, 32 splits, more splits than tiles) and its PDL predecessor's row
    "test_gpu_attention_aimed.py": "(varlen and (5-1-d128-tc5-bf16 or 4-1-d64-wmma64-bf16)) or (decode_aimed and 8-2-d64-16 and bf16) or pdl",
    # the W4A16 prefill GEMM against the dense GEMM, bit for bit, at the small shapes (every epilogue, split-K, both dtypes), and its checks
    "test_gpu_w4_prefill.py": "small or bad_arguments",
}

# --quick: a subset that finishes in about a minute (what tests/test_shim_kernels.py runs inside the CPU suite)
QUICK = {
    "test_gpu_zz_b_sampling.py": "matches_reference and (1000 or 4096)",
    "test_gpu_zz_c_train.py": "adamw_and_clip or lora_pack or (test_attention_backward and (lens1 or lens4 or gqa)) or (train_step_matches_oracle and True-64)",
    "test_gpu_train_kernels.py": None,
    "test_gpu_zz_e_fused_decode.py": None,
    "test_gpu_gemm.py": "not deterministic_under_repetition",
    "test_gpu_zz_d_attn_bwd_tc5.py": "lens0 or lens1 or lens4",
    # the two kernels of round 2's second session: the persistent single-pass prefill attention (the lazy-rescale and the many-items cases)
    # and the W4A16 mma kernel (two small shapes, both dtypes)
    "test_gpu_attention.py": "growing or many_items",
    "test_gpu_w4.py": "mma_partials and (256-512-128-5-2 or 528-1536)",
}

if __name__ == "__main__":
    extra = sys.argv[1:]
    if "--quick" in extra:
        extra.remove("--quick")
        SELECT = QUICK
    print("entry points running from kernel source:", " ".join(sorted(_shim_native)))
    rc = 0
    for f, k in SELECT.items():
        args = [os.path.join(ROOT, "tests", f), "-q", "-p", "no:cacheprovider", "--runxfail", "-m", "gpu", "-x"] + (["-k", k] if k and "-k" not in extra else []) + extra
        rc |= int(pytest.main(args))
    sys.exit(rc)
