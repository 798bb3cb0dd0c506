#!/usr/bin/env python
"""Dry run of the benchmark drivers on a machine WITHOUT a GPU (TEST INFRASTRUCTURE ONLY -- not a measurement).

    python tools/dryrun_bench.py decode [bench.py flags]      # bench.py's B200 arm
    python tools/dryrun_bench.py lora                         # tools/bench_lora.py

The C-ABI is replaced by the torch test double (tests/cabi_double.py), `device="cuda"` is dropped, CUDA events / graphs / clock
sampling are stubs, and the model is shrunk to toy dimensions.  What this exercises is the DRIVER LOGIC the round-end run depends
on -- batch assembly, prefill + decode loop, launch counting, the roofline / attention / TS-encoder side measurements, the e2e leg
and the JSON line -- so that a Python-level mistake in a script that only ever runs on the GPU box is caught here.  The numbers
it prints are meaningless."""
import contextlib
import functools
import importlib.util
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def _strip_cuda():
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
    _to = torch.Tensor.to

    def to(self, *a, **k):
        a = tuple(x for x in a if not (isinstance(x, (str, torch.device)) and "cuda" in str(x)))
        if "cuda" in str(k.get("device", "")):
            k.pop("device")
        k.pop("non_blocking", None)
        return _to(self, *a, **k) if (a or k) else self
    torch.Tensor.to = to
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.Tensor.pin_memory = lambda self: self
    torch.cuda.synchronize = lambda *a, **k: None
    torch.cuda.is_available = lambda: True
    torch.cuda.current_device = lambda: 0
    torch.cuda.set_device = lambda *a: None
    torch.cuda.is_current_stream_capturing = lambda: False

    class Event:
        def __init__(self, **k):
            self.t = 0.0

        def record(self, *a):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3

    class Graph:
        def replay(self):
            pass
    torch.cuda.Event = Event
    torch.cuda.CUDAGraph = Graph
    torch.cuda.graph = lambda g, **k: contextlib.nullcontext()


def _install_double():
    from tests.cabi_double import TorchDouble
    from chatts_b200 import _cabi
    import chatts_b200.model as mm
    import chatts_b200.ts_encoder as te
    dbl = TorchDouble()
    dbl.arch = "double"
    _cabi.get_context = lambda device=None: dbl
    init = mm.ChatTSForCausalLM.__init__

    def _init(self, config, state_dict, device="cpu", **kw):
        kw["use_cuda_graph"] = False
        init(self, config, state_dict, device="cpu", **kw)
    mm.ChatTSForCausalLM.__init__ = _init
    fs = mm.ChatTSForCausalLM.from_synthetic.__func__
    mm.ChatTSForCausalLM.from_synthetic = classmethod(
        lambda cls, config=None, seed=1234, device="cpu", dtype=torch.bfloat16, gen_device=None, **kw: fs(cls, config, seed, "cpu", dtype, "cpu", **kw))
    te_init = te.TimeSeriesEmbedding.__init__
    te.TimeSeriesEmbedding.__init__ = lambda self, config, weights, device="cpu", **kw: te_init(self, config, weights, device="cpu", **kw)


class _Clocks:
    def __init__(self, *a):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def summary(self):
        return {"sm_mhz": 0, "sm_max_mhz": 0, "reasons": []}


def _toy(factory, layers):
    def small():
        c = factory()
        c.hidden_size, c.intermediate_size, c.num_attention_heads, c.num_key_value_heads, c.head_dim = 256, 512, 4, 2, 64
        c.num_hidden_layers = layers
        c.ts["hidden_size"] = 256
        return c
    return staticmethod(small)


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "decode"
    _strip_cuda()
    _install_double()
    import bench
    from chatts_b200 import ChatTSConfig
    bench.ClockSampler = _Clocks
    if which == "decode":
        ChatTSConfig.chatts_14b = _toy(ChatTSConfig.chatts_14b, 2)
        sys.argv = ["bench.py", "--steps", "2", "--warmup", "1", "--batch", "2", "--no-cpu-baseline"] + sys.argv[2:]      # later flags win
        bench.main()
    else:
        ChatTSConfig.chatts_8b = _toy(ChatTSConfig.chatts_8b, 1)
        spec = importlib.util.spec_from_file_location("bench_lora", os.path.join(ROOT, "tools", "bench_lora.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        m.ClockSampler = _Clocks
        sys.argv = ["bench_lora.py", "--steps", "1", "--warmup", "1", "--samples", "1"]
        m.main()


if __name__ == "__main__":
    main()
