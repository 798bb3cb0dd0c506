"""OpenAI-style HTTP front end for the B200 engine (SURVEY.md 8(f) N3): what ``scripts/start_vllm_server.sh`` +
``demo/vllm_api.py`` give a ChatTS user -- ``POST /v1/chat/completions`` whose user message carries text parts and
``{"timeseries": [...]}`` parts, consumed in ``<ts><ts/>`` order (demo/vllm_api.py:45-55) -- plus ``/v1/completions`` with the
vLLM request shape (``prompt`` + ``multi_modal_data.timeseries``, demo/demo_vllm.py:47-52), ``/v1/models`` and ``/health``.

    python -m chatts_b200.server --model /path/to/ChatTS-14B --port 12345
    client = openai.OpenAI(base_url="http://127.0.0.1:12345/v1", api_key="test")        # demo/vllm_api.py works unchanged

Scheduling: ONE worker thread owns the model (one host thread per C-ABI context).  Requests that arrive within
``batch_window_ms`` of each other and share their sampling parameters are decoded as one batch (up to ``max_num_seqs``) --
static micro-batching, a batch runs to completion before the next one starts (``--scheduler batch``, sampling supported); or
iteration-level batching over the static decode slots (``--scheduler continuous``, engine.ContinuousEngine: requests join and
leave between graph replays; greedy).  ``stream=true`` sends one SSE chunk per generated token through the engine's streamer hook.
Host-side plumbing only: every number comes from ``vllm_compat.LLM`` -> ``ChatTSForCausalLM`` -> libchatts_b200.so.
"""
import argparse
import json
import queue
import threading
import time
import uuid
from concurrent.futures import Future
from dataclasses import dataclass, field

from .vllm_compat import IncrementalDecoder, eos_ids

MAX_TS_DEFAULT = 15          # scripts/start_vllm_server.sh:9  (--limit-mm-per-prompt timeseries=15)


@dataclass
class _Job:
    prompt: str
    series: list
    params: dict
    future: Future = field(default_factory=Future)
    stream_q: "queue.Queue | None" = None


def messages_to_prompt(messages, tokenizer=None, chat_template=True):
    """OpenAI chat messages -> (prompt text, series list).  Text parts are concatenated in order, ``{"timeseries": [...]}``
    parts are collected in order (they pair with the ``<ts><ts/>`` placeholders of the text, demo/vllm_api.py:36,52).  With a
    tokenizer that has a chat template and ``chat_template=True`` the roles are rendered by it; otherwise the ChatML layout
    the reference's demos write by hand (demo/vllm_api.py:37) is used unless the text already contains ``<|im_start|>``."""
    series, turns = [], []
    for m in messages:
        content = m.get("content", "")
        if isinstance(content, str):
            text = content
        else:
            text = ""
            for part in content:
                if "timeseries" in part:
                    series.append(part["timeseries"])
                elif part.get("type") == "text" or "text" in part:
                    text += part.get("text", "")
                else:
                    raise ValueError(f"unsupported content part: {sorted(part)}")
        turns.append({"role": m.get("role", "user"), "content": text})
    if len(turns) == 1 and "<|im_start|>" in turns[0]["content"]:
        return turns[0]["content"], series                      # the caller templated the prompt itself (demo/vllm_api.py:37)
    if chat_template and tokenizer is not None and getattr(tokenizer, "chat_template", None):
        return tokenizer.apply_chat_template(turns, add_generation_prompt=True, tokenize=False), series
    out = "".join(f"<|im_start|>{t['role']}\n{t['content']}<|im_end|>" for t in turns) + "<|im_start|>assistant\n"
    return out, series


class Engine:
    """Worker thread + request queue around a ``vllm_compat.LLM``."""

    def __init__(self, llm, batch_window_ms=5.0, max_ts_per_prompt=MAX_TS_DEFAULT, scheduler="batch", steps_per_round=4, autostart=True):
        self.llm, self.window, self.max_ts = llm, batch_window_ms / 1e3, max_ts_per_prompt
        self.q = queue.Queue()
        self.stop = False
        self.batches = []                                 # sizes of the batches run so far (observability / tests)
        self.scheduler, self.steps_per_round = scheduler, steps_per_round
        self.occupancy = []                               # continuous scheduler: active slots per round
        self.thread = threading.Thread(target=self._loop_continuous if scheduler == "continuous" else self._loop, daemon=True)
        if autostart:
            self.thread.start()

    def start(self):
        """Start the worker (``autostart=False`` lets a caller queue requests first: deterministic batches in tests)."""
        if not self.thread.is_alive():
            self.thread.start()

    def submit(self, prompt, series, params, stream=False):
        if len(series) > self.max_ts:
            raise ValueError(f"at most {self.max_ts} time series per prompt")
        if self.scheduler == "continuous" and params.get("temperature", 0.0) > 0:
            raise ValueError("the continuous scheduler decodes greedily; start the server with --scheduler batch for sampling")
        job = _Job(prompt, list(series), dict(params), stream_q=queue.Queue() if stream else None)
        self.q.put(job)
        return job

    def close(self):
        self.stop = True
        self.q.put(None)
        if self.thread.is_alive():
            self.thread.join(timeout=10)

    # -------------------------------------------------------------------------------------------- worker
    def _loop(self):
        from .vllm_compat import SamplingParams
        while not self.stop:
            job = self.q.get()
            if job is None:
                break
            batch = [job]
            deadline = time.monotonic() + self.window
            cap = self.llm.model.max_batch
            while len(batch) < cap and job.stream_q is None:
                try:
                    nxt = self.q.get(timeout=max(0.0, deadline - time.monotonic()))
                except queue.Empty:
                    break
                if nxt is None:
                    self.stop = True
                    break
                if nxt.params == job.params and nxt.stream_q is None:
                    batch.append(nxt)
                else:
                    self.q.put(nxt)                       # different sampling parameters / streaming: its own batch, next round
                    break
            self.batches.append(len(batch))
            try:
                sp = SamplingParams(**job.params)
                reqs = [{"prompt": j.prompt, "multi_modal_data": {"timeseries": j.series}} if j.series else {"prompt": j.prompt} for j in batch]
                if job.stream_q is not None:
                    gd = getattr(self.llm.model, "generation_defaults", None) or {}
                    stop_ids = [] if sp.ignore_eos else eos_ids(self.llm.model.config, sp.stop_token_ids, gd.get("eos_token_id"))
                    outs = self.llm.generate(reqs, sp, streamer=_QueueStreamer(job.stream_q, self.llm.tokenizer, stop_ids))
                else:
                    outs = self.llm.generate(reqs, sp)
                for j, o in zip(batch, outs):
                    j.future.set_result(o)
            except Exception as e:      # surfaced to every caller of the batch; the worker keeps serving
                for j in batch:
                    if not j.future.done():
                        j.future.set_exception(e)
            finally:
                if job.stream_q is not None:
                    job.stream_q.put(None)


    # -------------------------------------------------------------------------------------------- continuous scheduler
    def _loop_continuous(self):
        """Iteration-level batching (engine.ContinuousEngine): requests join the static decode slots between graph replays and
        leave them at EOS / max_tokens; streaming requests get their new tokens after every round."""
        from .engine import ContinuousEngine
        from .vllm_compat import CompletionOutput, RequestOutput, cut_at_stop, cut_at_stop_string, decode_text
        llm = self.llm
        eng = ContinuousEngine(llm.model, steps_per_round=self.steps_per_round)
        jobs, sent = {}, {}

        def admit(job):
            try:
                enc = llm.processor(text=[job.prompt], timeseries=job.series, padding=True, return_tensors="pt")
                p = job.params
                gd = getattr(llm.model, "generation_defaults", None) or {}
                job.stop_ids = eos_ids(llm.model.config, p.get("stop_token_ids"), gd.get("eos_token_id"))
                rid = eng.add_request(enc["input_ids"][0], enc["timeseries"], max_new_tokens=p.get("max_tokens", 16),
                                      eos_token_id=job.stop_ids, ignore_eos=p.get("ignore_eos", False))
                jobs[rid], sent[rid] = job, 0
                if job.stream_q is not None:
                    job.decoder = IncrementalDecoder(llm.tokenizer)
            except Exception as e:
                job.future.set_exception(e)
                if job.stream_q is not None:
                    job.stream_q.put(None)

        def finish(job, tokens):
            toks, fin = cut_at_stop(tokens, job.stop_ids, job.params.get("ignore_eos", False))
            text, hit = cut_at_stop_string(decode_text(llm.tokenizer, toks), job.params.get("stop") or [])
            return CompletionOutput(text, toks, "stop" if hit else fin)

        while not self.stop:
            if not eng.has_work():
                job = self.q.get()
                if job is None:
                    break
                admit(job)
            while True:
                try:
                    job = self.q.get_nowait()
                except queue.Empty:
                    break
                if job is None:
                    self.stop = True
                    break
                admit(job)
            try:
                finished = eng.step()
            except Exception as e:      # an engine failure ends every request in flight; the loop keeps serving new ones
                for rid, job in list(jobs.items()):
                    if not job.future.done():
                        job.future.set_exception(e)
                    if job.stream_q is not None:
                        job.stream_q.put(None)
                jobs.clear(); sent.clear()
                continue
            if eng.occupancy:
                self.occupancy.append(eng.occupancy[-1])
            for r in list(eng.active.values()) + list(finished):       # streaming: hand over what the round produced
                job = jobs.get(r.rid)
                if job is not None and job.stream_q is not None:
                    new, _ = cut_at_stop(r.tokens, job.stop_ids, job.params.get("ignore_eos", False))
                    piece = job.decoder.push(new[sent[r.rid]:])          # cumulative decode, new suffix only; the stop token is never streamed
                    if piece:
                        job.stream_q.put(piece)
                    sent[r.rid] = len(new)
            for r in finished:
                job = jobs.pop(r.rid, None)
                sent.pop(r.rid, None)
                if job is None:
                    continue
                if r.error is not None:                       # not admitted (over-long prompt, series mismatch, larger than the pool)
                    job.future.set_exception(r.error)
                    if job.stream_q is not None:
                        job.stream_q.put(None)
                    continue
                n = max(1, int(job.params.get("n", 1)))
                out = finish(job, r.tokens)
                job.future.set_result(RequestOutput(job.prompt, [out] * n))
                if job.stream_q is not None:
                    tail = job.decoder.flush()
                    if tail:
                        job.stream_q.put(tail)
                    job.stream_q.put(None)
        eng.close()


class _QueueStreamer:
    """HF-streamer protocol (put / end) -> per-token text pieces on a queue (single-request batches)."""

    def __init__(self, q, tokenizer, stop_ids=()):
        self.q, self.dec, self.stop, self.ended = q, IncrementalDecoder(tokenizer), set(int(t) for t in stop_ids), False

    def put(self, ids):
        t = int(ids.reshape(-1)[0])
        if self.ended or t in self.stop:          # the stop token (and the pad fill after it) is not text
            self.ended = True
            return
        piece = self.dec.push([t])                # cumulative decode: multi-byte characters arrive whole
        if piece:
            self.q.put(piece)

    def end(self):
        tail = self.dec.flush()
        if tail:
            self.q.put(tail)


def _sampling_from_body(body):
    p = {"max_tokens": int(body.get("max_tokens") or body.get("max_completion_tokens") or 256),
         "temperature": float(body.get("temperature", 0.0) or 0.0), "top_p": float(body.get("top_p", 1.0) or 1.0),
         "top_k": int(body.get("top_k", 0) or 0), "n": int(body.get("n", 1) or 1)}
    stop = body.get("stop")
    if stop:
        p["stop"] = [stop] if isinstance(stop, str) else list(stop)
    if body.get("stop_token_ids"):
        p["stop_token_ids"] = list(body["stop_token_ids"])
    if body.get("seed") is not None:
        p["seed"] = int(body["seed"])
    if body.get("ignore_eos"):
        p["ignore_eos"] = True
    return p


def create_app(llm, served_model_name="chatts", batch_window_ms=5.0, max_ts_per_prompt=MAX_TS_DEFAULT, scheduler="batch",
               steps_per_round=4):
    from fastapi import FastAPI, HTTPException, Request
    from fastapi.responses import JSONResponse, StreamingResponse

    app = FastAPI(title="chatts_b200")
    engine = Engine(llm, batch_window_ms, max_ts_per_prompt, scheduler, steps_per_round)
    app.state.engine = engine

    @app.get("/health")
    def health():
        return {"status": "ok"}

    @app.get("/v1/models")
    def models():
        return {"object": "list", "data": [{"id": served_model_name, "object": "model", "owned_by": "chatts_b200"}]}

    def usage(prompt, outs):
        n_out = sum(len(c.token_ids) for c in outs)
        n_in = len(llm.tokenizer.encode(prompt)) if hasattr(llm.tokenizer, "encode") else 0
        return {"prompt_tokens": n_in, "completion_tokens": n_out, "total_tokens": n_in + n_out}

    async def run(prompt, series, body, chat):
        import asyncio
        params = _sampling_from_body(body)
        rid = ("chatcmpl-" if chat else "cmpl-") + uuid.uuid4().hex[:24]
        created = int(time.time())
        n_ph = prompt.count("<ts><ts/>")
        if n_ph != len(series):                                      # the reference asserts the same (encoding_utils.py:58,68)
            raise HTTPException(400, f"{n_ph} <ts><ts/> placeholders but {len(series)} time series")
        try:
            job = engine.submit(prompt, series, params, stream=bool(body.get("stream")))
        except ValueError as e:
            raise HTTPException(400, str(e))
        if body.get("stream"):
            def gen():
                first = True
                while True:
                    piece = job.stream_q.get()
                    if piece is None:
                        break
                    delta = {"role": "assistant", "content": piece} if (chat and first) else ({"content": piece} if chat else None)
                    first = False
                    ch = {"index": 0, "delta": delta, "finish_reason": None} if chat else {"index": 0, "text": piece, "finish_reason": None}
                    yield "data: " + json.dumps({"id": rid, "object": "chat.completion.chunk" if chat else "text_completion", "created": created,
                                                 "model": served_model_name, "choices": [ch]}) + "\n\n"
                ch = {"index": 0, "delta": {}, "finish_reason": "stop"} if chat else {"index": 0, "text": "", "finish_reason": "stop"}
                yield "data: " + json.dumps({"id": rid, "object": "chat.completion.chunk" if chat else "text_completion", "created": created,
                                             "model": served_model_name, "choices": [ch]}) + "\n\n"
                yield "data: [DONE]\n\n"
            return StreamingResponse(gen(), media_type="text/event-stream")
        try:
            out = await asyncio.wrap_future(job.future)
        except (AssertionError, TypeError, ValueError) as e:         # the reference's own input errors (encoding_utils.py:58,68; chatts_vllm.py:277)
            raise HTTPException(400, str(e))
        choices = []
        for i, c in enumerate(out.outputs):
            fin = c.finish_reason or ("length" if len(c.token_ids) >= params["max_tokens"] else "stop")
            choices.append({"index": i, "message": {"role": "assistant", "content": c.text}, "finish_reason": fin} if chat else
                           {"index": i, "text": c.text, "finish_reason": fin})
        return JSONResponse({"id": rid, "object": "chat.completion" if chat else "text_completion", "created": created,
                             "model": served_model_name, "choices": choices, "usage": usage(prompt, out.outputs)})

    @app.post("/v1/chat/completions")
    async def chat_completions(request: Request):
        body = await request.json()
        try:
            prompt, series = messages_to_prompt(body.get("messages", []), llm.tokenizer)
        except ValueError as e:
            raise HTTPException(400, str(e))
        return await run(prompt, series, body, chat=True)

    @app.post("/v1/completions")
    async def completions(request: Request):
        body = await request.json()
        prompt = body.get("prompt", "")
        series = (body.get("multi_modal_data") or {}).get("timeseries", [])
        return await run(prompt, series, body, chat=False)

    return app


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default=None, help="checkpoint directory; default: synthetic ChatTS-14B weights + byte tokenizer")
    ap.add_argument("--served-model-name", default="chatts")
    ap.add_argument("--host", default="0.0.0.0")
    ap.add_argument("--port", type=int, default=12345)
    ap.add_argument("--max-model-len", type=int, default=6000)
    ap.add_argument("--max-num-seqs", type=int, default=32)
    ap.add_argument("--limit-mm-per-prompt", default="timeseries=15")
    ap.add_argument("--dtype", default="bfloat16")
    ap.add_argument("--batch-window-ms", type=float, default=5.0)
    ap.add_argument("--scheduler", default="batch", choices=["batch", "continuous"],
                    help="batch: micro-batches run to completion (sampling supported); continuous: iteration-level batching, greedy")
    ap.add_argument("--steps-per-round", type=int, default=4, help="continuous scheduler: decode steps between two host reads")
    ap.add_argument("--w4-only", action="store_true",
                    help="GPTQ-Int4 checkpoint: keep the decoder projections as 4-bit weights only (no dense copy; frees HBM for KV cache)")
    args = ap.parse_args()
    import uvicorn
    from .vllm_compat import LLM
    limit = int(dict(kv.split("=") for kv in args.limit_mm_per_prompt.split(",")).get("timeseries", MAX_TS_DEFAULT))
    tok = None
    if args.model:
        from transformers import AutoTokenizer
        tok = AutoTokenizer.from_pretrained(args.model, trust_remote_code=True)
    llm = LLM(model=args.model, tokenizer=tok, dtype=args.dtype, max_model_len=args.max_model_len, max_num_seqs=args.max_num_seqs,
              limit_mm_per_prompt={"timeseries": limit}, w4_only=args.w4_only)
    uvicorn.run(create_app(llm, args.served_model_name, args.batch_window_ms, limit, args.scheduler, args.steps_per_round),
                host=args.host, port=args.port)


if __name__ == "__main__":
    main()
