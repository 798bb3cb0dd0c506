"""TEST INFRASTRUCTURE ONLY -- what the tests of cts_gemm_w4_prefill need on a machine without a GPU:

  * ``add_w4_prefill(double)``: gives a tests/cabi_double.TorchDouble instance the entry point, answered by cts_gemm's double on the
    dense weight that the double's own fragment-major decoder (its gemm_w4_mma) recovers -- decoded once per weight tensor;
  * ``shim_context_w4p()``: the CUDA-on-CPU shim library of tests/cuda_on_cpu with csrc/gemm_w4_persistent.cu compiled in as well, built
    into a directory of its own so the standard shim library is left as it is."""
import os
import types

import torch

W4P_SOURCE = "gemm_w4_persistent.cu"


def _dense_weight(dbl, qwf, szp, n, group_size, dtype):
    """W [n, k] from the fragment-major copy: gemm_w4_mma of the k x k identity is W^T, exactly (each output is one product 1 * w)."""
    k = szp.shape[1] * int(group_size)
    key = (qwf.data_ptr(), szp.data_ptr(), int(n), int(group_size), dtype)
    cache = dbl.__dict__.setdefault("_w4p_cache", {})
    if key not in cache:
        out = torch.zeros(1, k, int(n))
        dbl.gemm_w4_mma(torch.eye(k, dtype=dtype), qwf, szp, n, group_size, out, 1, t=k)
        cache[key] = out[0].t().contiguous().to(dtype)
    return cache[key]


def _gemm_w4_prefill(self, x, qwf, szp, n, group_size, out, *, bias=None, residual=None, epilogue=0, split_k=1, t=None):
    """cts_gemm_w4_prefill: cts_gemm's epilogue over the dequantised weight, with the preconditions of cts_gemm_w4p_args."""
    k = szp.shape[1] * int(group_size)
    t = x.shape[0] if t is None else t
    assert k % 128 == 0 and (int(group_size) == 64 or int(group_size) % 128 == 0) and 1 <= split_k <= k // 64
    assert epilogue in (0, 3, 4, 6) and (split_k == 1 or epilogue == 3)
    assert epilogue != 6 or (int(n) % 128 == 0 and t > 128)
    w = _dense_weight(self, qwf, szp, n, group_size, x.dtype)
    self.gemm(x, w, out, bias=bias, residual=residual, epilogue=epilogue, split_k=split_k, t=t)


def add_w4_prefill(dbl):
    dbl.gemm_w4_prefill = types.MethodType(_gemm_w4_prefill, dbl)
    return dbl


def shim_context_w4p():
    import tests.cuda_on_cpu.build as sb
    from tests.cuda_on_cpu.shim import shim_context
    saved = sb.SOURCES, sb.OUT
    sb.SOURCES = list(saved[0]) + ([W4P_SOURCE] if W4P_SOURCE not in saved[0] else [])
    sb.OUT = os.path.join(os.path.dirname(saved[1]), "w4p", os.path.basename(saved[1]))
    try:
        return shim_context()
    finally:
        sb.SOURCES, sb.OUT = saved
