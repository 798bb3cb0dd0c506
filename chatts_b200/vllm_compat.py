"""Request/response shim for the vLLM surface of the reference (demo/demo_vllm.py:18-63,
chatts/utils/llm_utils.py:147-190): ``LLM(model=...).generate([{"prompt": str, "multi_modal_data":
{"timeseries": [...]}}], SamplingParams(...)) -> outputs[i].outputs[0].text``.

The reference's plugin file targets vllm 0.8.5 internals that no longer exist (SURVEY.md §8b); this shim
keeps the REQUEST SHAPE and drives the B200 engine directly instead of vLLM's plugin ABI."""
from dataclasses import dataclass, field

import numpy as np
import torch

from .config import ChatTSConfig
from .model import ChatTSForCausalLM
from .processor import ChatTSProcessor, SimpleTokenizer

MAX_TS_PER_PROMPT = 50      # chatts_vllm.py:219-220


@dataclass
class SamplingParams:
    """The fields the reference's callers set (llm_utils.py:153: temperature, top_p, max_tokens, stop_token_ids, stop, n;
    demo/demo_vllm.py:24)."""
    max_tokens: int = 16
    temperature: float = 0.0
    top_p: float = 1.0
    top_k: int = 0
    stop_token_ids: list = field(default_factory=list)
    stop: list = field(default_factory=list)          # stop STRINGS: the text is cut before the first occurrence
    n: int = 1                                        # completions per request (temperature > 0: independent seeds)
    ignore_eos: bool = False
    seed: int = None
    repetition_penalty: float = 1.0                   # vLLM SamplingParams.repetition_penalty (prompt + generated tokens)


@dataclass
class CompletionOutput:
    text: str
    token_ids: list
    finish_reason: str = None     # "stop" (EOS / stop id / stop string) or "length"


def eos_ids(config, stop_token_ids=None, extra=None):
    """Stop ids of a request: the UNION of the model's EOS ids (config / generation_config) and the request's stop_token_ids
    (vLLM adds stop_token_ids to the EOS stop, it does not replace it; llm_utils.py:153 passes both Qwen ids explicitly)."""
    out = []
    for src in (getattr(config, "eos_token_id", None), extra, stop_token_ids):
        if src is None:
            continue
        out += [int(t) for t in (src if isinstance(src, (list, tuple, set)) else [src])]
    return sorted(set(out))


def cut_at_stop(tokens, stop_ids, ignore_eos=False):
    """(tokens before the first stop id, finish_reason).  The stop token itself is not part of the completion (vLLM strips it; the
    reference decodes with skip_special_tokens=True); whatever generate() padded a finished row with is dropped with it."""
    toks = [int(t) for t in tokens]
    if not ignore_eos:
        stop = set(int(t) for t in stop_ids)
        for i, t in enumerate(toks):
            if t in stop:
                return toks[:i], "stop"
    return toks, "length"


def decode_text(tokenizer, tokens):
    """tokenizer.decode(..., skip_special_tokens=True) (inference_tsmllm_deepspeed.py:104-106), for tokenizers that take the flag."""
    try:
        return tokenizer.decode(tokens, skip_special_tokens=True)
    except TypeError:
        return tokenizer.decode(tokens)


def cut_at_stop_string(text, stops):
    cut = min([text.find(st) for st in stops if st and st in text], default=-1)
    return (text[:cut], True) if cut >= 0 else (text, False)


class IncrementalDecoder:
    """Streaming detokeniser: decodes the CUMULATIVE ids and emits only the new suffix, holding back a trailing U+FFFD (an
    incomplete multi-byte character, e.g. half of a Chinese character) until the bytes that complete it arrive."""

    def __init__(self, tokenizer):
        self.tok, self.ids, self.sent = tokenizer, [], 0

    def push(self, token_ids):
        self.ids += [int(t) for t in token_ids]
        text = decode_text(self.tok, self.ids)
        while text.endswith("\ufffd"):
            text = text[:-1]
        piece = text[self.sent:]
        self.sent = max(self.sent, len(text))
        return piece

    def flush(self):
        text = decode_text(self.tok, self.ids)
        piece = text[self.sent:]
        self.sent = len(text)
        return piece


@dataclass
class RequestOutput:
    prompt: str
    outputs: list


def _free_port():
    import socket
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0))
        return so.getsockname()[1]


def _tp_worker(rank, world, port, backend, factory, factory_kw):
    """Body of a spawned tensor-parallel rank (rank >= 1): join the group, build the same engine on this rank's shard, then mirror
    every call the driver (rank 0) broadcasts -- the ranks of a tensor-parallel model run the same program (SPMD)."""
    import os
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    else:
        dist.init_process_group(backend, rank=rank, world_size=world)
    engine = factory(**factory_kw)
    while True:
        box = [None]
        dist.broadcast_object_list(box, src=0)
        cmd = box[0]
        if cmd[0] == "stop":
            break
        if cmd[0] == "generate":
            engine._generate(cmd[1], cmd[2])
    dist.destroy_process_group()


def _make_llm(**kw):
    return LLM(**kw)


class LLM:
    def __init__(self, model=None, tokenizer=None, config=None, state_dict=None, tensor_parallel_size=1, dtype="bfloat16",
                 max_model_len=2048, max_num_seqs=32, limit_mm_per_prompt=None, trust_remote_code=True, seed=1234,
                 distributed_backend="nccl", w4_only=False, **kw):
        """tensor_parallel_size = k > 1 (every caller of the reference passes it: demo/demo_vllm.py:30, llm_utils.py:153-154):
          * under torchrun / an initialised process group of k ranks the engine ATTACHES: every rank constructs the LLM and makes the
            same generate() calls (rank r holds shard r);
          * otherwise the constructor SPAWNS k - 1 worker processes (one per GPU, as vLLM's multiprocessing executor does,
            README.md:141) that build their shards and mirror every generate() call of this process (rank 0) -- the model must then
            be named by a path or by config + seed (a ChatTSForCausalLM instance cannot be sent to another process).
        w4_only=True: a GPTQ-Int4 checkpoint path is loaded with its projections as 4-bit weights only (from_pretrained(w4_only=True))."""
        import os
        self._tp_procs, self._tp_driver = [], False
        tp = int(tensor_parallel_size or 1)
        tp_kw = {}
        if tp > 1:
            import torch.distributed as dist
            attach = dist.is_available() and dist.is_initialized()
            if not attach and int(os.environ.get("WORLD_SIZE", "1")) == tp:          # torchrun started us: join its group
                local = int(os.environ.get("LOCAL_RANK", "0"))
                if distributed_backend == "nccl":
                    torch.cuda.set_device(local)
                    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
                else:
                    dist.init_process_group(distributed_backend)
                attach = True
            if attach:
                if dist.get_world_size() != tp:
                    raise ValueError(f"tensor_parallel_size={tp} but the process group has {dist.get_world_size()} ranks")
                tp_kw = dict(tp_rank=dist.get_rank(), tp_size=tp)
            else:
                if isinstance(model, ChatTSForCausalLM) or state_dict is not None:
                    raise ValueError("spawning tensor-parallel ranks needs a model PATH or config + seed (launch with torchrun to pass "
                                     "a constructed model or a state dict on every rank)")
                import torch.multiprocessing as mp
                port = _free_port()
                child_kw = dict(model=model, tokenizer=tokenizer, config=config, tensor_parallel_size=tp, dtype=dtype, max_model_len=max_model_len,
                                max_num_seqs=max_num_seqs, limit_mm_per_prompt=limit_mm_per_prompt, seed=seed,
                                distributed_backend=distributed_backend, **kw)
                ctx = mp.get_context("spawn")
                for r in range(1, tp):
                    pr = ctx.Process(target=_tp_worker, args=(r, tp, port, distributed_backend, _make_llm, child_kw), daemon=True)
                    pr.start()
                    self._tp_procs.append(pr)
                os.environ.update(RANK="0", LOCAL_RANK="0", WORLD_SIZE=str(tp), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
                if distributed_backend == "nccl":
                    torch.cuda.set_device(0)
                    dist.init_process_group("nccl", rank=0, world_size=tp, device_id=torch.device("cuda:0"))
                else:
                    dist.init_process_group(distributed_backend, rank=0, world_size=tp)
                self._tp_driver = True
                tp_kw = dict(tp_rank=0, tp_size=tp)
        dt = torch.bfloat16 if str(dtype) in ("bfloat16", "torch.bfloat16") else torch.float16
        if isinstance(model, ChatTSForCausalLM):
            self.model = model
        elif isinstance(model, str):
            self.model = ChatTSForCausalLM.from_pretrained(model, torch_dtype=dt, max_seq_len=max_model_len, max_batch=max_num_seqs,
                                                           w4_only=w4_only, **tp_kw)
        else:
            cfg = config or ChatTSConfig.chatts_14b()
            self.model = (ChatTSForCausalLM(cfg, state_dict, dtype=dt, max_seq_len=max_model_len, max_batch=max_num_seqs, **tp_kw)
                          if state_dict is not None else
                          ChatTSForCausalLM.from_synthetic(cfg, seed=seed, dtype=dt, max_seq_len=max_model_len, max_batch=max_num_seqs, **tp_kw))
        cfg = self.model.config
        self.tokenizer = tokenizer or SimpleTokenizer(cfg.ts_token_start_index, cfg.pad_token_id, cfg.eos_token_id)
        self.processor = ChatTSProcessor(self.tokenizer, cfg, dtype=torch.float32)
        self.limit = (limit_mm_per_prompt or {}).get("timeseries", MAX_TS_PER_PROMPT)

    def shutdown(self):
        """Stop the spawned tensor-parallel workers (no-op otherwise)."""
        if self._tp_driver:
            import torch.distributed as dist
            dist.broadcast_object_list([("stop",)], src=0)
            for pr in self._tp_procs:
                pr.join(timeout=30)
            dist.destroy_process_group()
            self._tp_driver, self._tp_procs = False, []

    def __del__(self):
        try:
            self.shutdown()
        except Exception:  # noqa: BLE001  (interpreter teardown)
            pass

    def generate(self, inputs, sampling_params=None, use_tqdm=False, streamer=None):
        sp = sampling_params or SamplingParams()
        if isinstance(inputs, (dict, str)):
            inputs = [inputs]
        # plain strings are text-only prompts (llm_utils.py:127 passes a list of str to the same call)
        inputs = [{"prompt": r} if isinstance(r, str) else r for r in inputs]
        n = max(1, int(sp.n))
        if n > 1:
            # n completions per request = n copies of the request in the batch, each row with its own draw
            # (llm_utils.py:127-130 reads outputs[i].outputs[j].text for j < n)
            flat = self._generate([r for r in inputs for _ in range(n)], sp)
            return [RequestOutput(inputs[i]["prompt"], [flat[i * n + j].outputs[0] for j in range(n)]) for i in range(len(inputs))]
        return self._generate(inputs, sp, streamer)

    def _generate(self, inputs, sp, streamer=None):
        if self._tp_driver:                                  # the spawned ranks run the same call on their shards
            import torch.distributed as dist
            dist.broadcast_object_list([("generate", inputs, sp)], src=0)
        outs = []
        bs = self.model.max_batch
        stops = [sp.stop] if isinstance(sp.stop, str) else list(sp.stop or [])
        gd = getattr(self.model, "generation_defaults", None) or {}
        stop_ids = eos_ids(self.model.config, sp.stop_token_ids, gd.get("eos_token_id"))
        for i0 in range(0, len(inputs), bs):
            chunk = inputs[i0:i0 + bs]
            prompts, series = [], []
            for req in chunk:
                ts = (req.get("multi_modal_data") or {}).get("timeseries", [])
                if len(ts) > self.limit:
                    raise ValueError(f"at most {self.limit} time series per prompt")
                for t in ts:
                    if not isinstance(t, (list, np.ndarray, torch.Tensor)):
                        raise TypeError(f"Unsupported time series type: {type(t)}")
                prompts.append(req["prompt"])
                series.extend(ts)
            enc = self.processor(text=prompts, timeseries=series, padding=True, return_tensors="pt")
            S = enc["input_ids"].shape[1]
            ids = self.model.generate(**enc, max_new_tokens=sp.max_tokens, do_sample=sp.temperature > 0,
                                      temperature=sp.temperature, top_p=sp.top_p, top_k=(sp.top_k if sp.top_k and sp.top_k > 0 else None),
                                      ignore_eos=sp.ignore_eos, seed=(None if sp.seed is None else sp.seed + i0),
                                      eos_token_id=stop_ids, streamer=streamer,
                                      repetition_penalty=(sp.repetition_penalty if sp.repetition_penalty not in (None, 1.0) else None))
            for b, req in enumerate(chunk):
                # a row ends at ITS first stop id (the batch-wide tail after it is the pad fill of generate())
                toks, fin = cut_at_stop(ids[b, S:].tolist(), stop_ids, sp.ignore_eos)
                text, hit = cut_at_stop_string(decode_text(self.tokenizer, toks), stops)
                outs.append(RequestOutput(req["prompt"], [CompletionOutput(text, toks, "stop" if hit else fin)]))
        return outs


# --------------------------------------------------------------------------------------------------
# Streaming surface of the reference's interactive script (chatts/utils/vllm_stream_qa.py:26-59):
#     model = AsyncLLMEngine.from_engine_args(AsyncEngineArgs(model=..., max_model_len=..., limit_mm_per_prompt={"timeseries": 15}))
#     async for request_output in model.generate(prompt, SamplingParams(max_tokens=...), request_id=...):
#         request_output.outputs[0].text            # CUMULATIVE text so far
# One request at a time per engine (the script is a chat loop); tokens come from the decode loop through the HF-streamer
# protocol of ChatTSForCausalLM.generate (put / end), one device->host read per token.
# --------------------------------------------------------------------------------------------------
@dataclass
class AsyncEngineArgs:
    model: object = None
    enforce_eager: bool = True                        # accepted and ignored: the decode step is always one CUDA graph
    gpu_memory_utilization: float = 0.9               # accepted and ignored: the KV pool is sized by max_model_len x max_num_seqs
    max_model_len: int = 2048
    tensor_parallel_size: int = 1
    limit_mm_per_prompt: dict = None
    trust_remote_code: bool = True
    dtype: str = "bfloat16"
    max_num_seqs: int = 1


class _AsyncStreamer:
    def __init__(self, loop, queue):
        self.loop, self.queue = loop, queue

    def put(self, ids):
        self.loop.call_soon_threadsafe(self.queue.put_nowait, [int(x) for x in ids.reshape(-1)[:1]])

    def end(self):
        pass


class AsyncLLMEngine:
    def __init__(self, llm):
        import threading
        self.llm = llm
        self._busy = threading.Lock()

    @classmethod
    def from_engine_args(cls, args, llm=None):
        if llm is None:
            llm = LLM(model=args.model, tensor_parallel_size=args.tensor_parallel_size, dtype=args.dtype, max_model_len=args.max_model_len,
                      max_num_seqs=args.max_num_seqs, limit_mm_per_prompt=args.limit_mm_per_prompt, trust_remote_code=args.trust_remote_code)
        return cls(llm)

    async def generate(self, prompt, sampling_params=None, request_id=None):
        """Async generator of RequestOutput with the cumulative text (and token ids) after every new token; the last one carries the
        final text with the stop strings applied, exactly what the blocking call returns."""
        import asyncio
        loop = asyncio.get_running_loop()
        q = asyncio.Queue()
        req = {"prompt": prompt} if isinstance(prompt, str) else prompt
        sp = sampling_params or SamplingParams()
        done = object()

        def work():
            with self._busy:
                try:
                    out = self.llm.generate([req], sp, streamer=_AsyncStreamer(loop, q))[0]
                    loop.call_soon_threadsafe(q.put_nowait, (done, out))
                except BaseException as e:          # surfaced in the consumer, not lost in the worker thread
                    loop.call_soon_threadsafe(q.put_nowait, (done, e))

        fut = loop.run_in_executor(None, work)
        toks = []
        stops = [sp.stop] if isinstance(sp.stop, str) else list(sp.stop or [])
        gd = getattr(self.llm.model, "generation_defaults", None) or {}
        stop_ids = set(eos_ids(self.llm.model.config, sp.stop_token_ids, gd.get("eos_token_id")))
        ended = False
        while True:
            item = await q.get()
            if isinstance(item, tuple) and item[0] is done:
                await fut
                if isinstance(item[1], BaseException):
                    raise item[1]
                yield item[1]
                return
            if ended or (not sp.ignore_eos and any(t in stop_ids for t in item)):
                ended = True                           # the stop token and anything after it never reach the stream
                continue
            toks += item
            text = decode_text(self.llm.tokenizer, toks)
            if any(st and st in text for st in stops):
                continue                               # the final output carries the text cut at the stop string
            if text.endswith("\ufffd"):
                continue                               # incomplete multi-byte character: wait for the bytes that complete it
            yield RequestOutput(req["prompt"], [CompletionOutput(text, list(toks))])
