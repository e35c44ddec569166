"""Optional HTTP front of a sampler engine with the wire format the reference's clients speak.

The reference's actor reaches its sampler over HTTP (vLLM's OpenAI-compatible server started by
pipelinerl/launch.py:191-247 / vllm1.py:189-273).  On one box this package talks to the engine in process
(serving.py), but REMOTE reference actors — or an unmodified `pipelinerl.async_llm.llm_async_generate` — can be pointed
at this shim instead of a vLLM server (SURVEY §8b "wire format"):

  POST /v1/chat/completions   request fields the reference sends (async_llm.py:96-131): model, messages, logprobs,
                              include_stop_str_in_output, skip_special_tokens, tools?, max_tokens?, chat_template_kwargs?
                              + llm.parameters (temperature, top_p, top_k ...);  response fields it reads (:173-207):
                              choices[0].message.{content, tool_calls}, choices[0].logprobs.content[i].{token, logprob}
                              with token = "token_id:<id>" (--return-tokens-as-token-ids), choices[0].finish_reason in
                              {stop, length}, usage.{prompt_tokens, completion_tokens}
  POST /v1/completions        the reference-logprob pass (llm.py:606-648): prompt = list of token-id lists, max_tokens 0,
                              echo true -> choices[i].prompt_logprobs = [None, {"<id>": {"logprob": ...}}, ...]
  GET  /health                200 once the engine thread is up (launch.py waits on it)
  POST /receive_weight_update the reference's trigger for its NCCL broadcast (vllm1.py:244-249).  Here weights arrive by
                              the learner's P2P push; the endpoint only reports the version the sampler is serving.

Sampling features the engine does not implement (n > 1, streaming; top_p < 1 and top_k > 0 unless the engine has
`supports_top_k_top_p`) are rejected with 400 rather than silently ignored, and so are top_p / top_k values vLLM would
reject (top_p outside (0, 1], top_k not an integer >= -1).  Host code only: the engine behind it is the CUDA
DecodeEngine (no CPU fallback).
"""
from __future__ import annotations

import asyncio
import queue
import time
import uuid
from typing import Any

from aiohttp import web

from .engine import SamplingParams


def _token_ids(encoded) -> list[int]:
    if hasattr(encoded, "keys") and "input_ids" in encoded.keys():
        encoded = encoded["input_ids"]
    return list(encoded)


class HttpShim:
    """server: an object with `async generate(prompt_ids, SamplingParams) -> request` (request has output_ids,
    output_logprobs, finish_reason, model_version), an `engine` with `score(list[list[int]], temperature)` and an
    `on_step_boundary` hook called on the engine thread (serving.EngineServer provides all three)."""

    def __init__(self, server, tokenizer, model_name: str, default_max_tokens: int = 16):
        self.server, self.tok, self.model_name = server, tokenizer, model_name
        self.default_max_tokens = default_max_tokens
        self._score_jobs: "queue.Queue[tuple]" = queue.Queue()
        prev = getattr(server, "on_step_boundary", None)

        def boundary(engine):
            if prev is not None:
                prev(engine)
            self._drain_score_jobs(engine)
        server.on_step_boundary = boundary
        self.app = web.Application()
        self.app.add_routes([web.post("/v1/chat/completions", self.chat_completions),
                             web.post("/v1/completions", self.completions),
                             web.get("/health", self.health),
                             web.post("/receive_weight_update", self.receive_weight_update)])
        self._runner: web.AppRunner | None = None
        self.port: int | None = None

    # ---- lifecycle ---------------------------------------------------------------------------
    async def start(self, host: str = "127.0.0.1", port: int = 0) -> str:
        self._runner = web.AppRunner(self.app)
        await self._runner.setup()
        site = web.TCPSite(self._runner, host, port)
        await site.start()
        self.port = site._server.sockets[0].getsockname()[1]
        return f"http://{host}:{self.port}"

    async def stop(self) -> None:
        if self._runner is not None:
            await self._runner.cleanup()

    # ---- engine-thread side of the scoring endpoint ---------------------------------------------
    def _drain_score_jobs(self, engine) -> None:
        while True:
            try:
                seqs, temperature, loop, fut = self._score_jobs.get_nowait()
            except queue.Empty:
                return
            try:
                res = engine.score(seqs, temperature)
                loop.call_soon_threadsafe(fut.set_result, res)
            except BaseException as e:  # noqa: BLE001  (forwarded to the waiting request)
                loop.call_soon_threadsafe(fut.set_exception, e)

    def _decode(self, ids: list[int]) -> str:
        if not ids:
            return ""
        try:
            return self.tok.decode(ids, skip_special_tokens=False)
        except TypeError:   # llm.SyntheticTokenizer: decode(ids)
            return self.tok.decode(ids)

    # ---- handlers ------------------------------------------------------------------------------
    @staticmethod
    def _bad(msg: str) -> web.Response:
        return web.json_response({"error": {"message": msg, "type": "invalid_request_error"}}, status=400)

    def _sampling(self, body: dict) -> SamplingParams | web.Response:
        top_k = -1 if body.get("top_k") is None else body["top_k"]          # null = vLLM's default
        top_p = 1.0 if body.get("top_p") is None else body["top_p"]
        try:
            filters = SamplingParams(top_k=top_k, top_p=top_p)
        except ValueError as e:
            return self._bad(str(e))
        if (top_p < 1.0 or top_k > 0) and not getattr(self.server.engine, "supports_top_k_top_p", False):
            return self._bad("top_p / top_k sampling is not implemented by this engine (the reference trains with "
                             "top_p=1, top_k=-1, conf/base.yaml:46-51)")
        if int(body.get("n", 1)) != 1 or body.get("stream"):
            return self._bad("n > 1 and streaming are not implemented")
        temperature = float(body.get("temperature", 1.0))
        max_tokens = int(body.get("max_tokens") or body.get("max_completion_tokens") or self.default_max_tokens)
        return SamplingParams(max_tokens=max_tokens, temperature=temperature if temperature > 0 else 1.0,
                              greedy=temperature <= 0, top_k=filters.top_k, top_p=filters.top_p)

    async def chat_completions(self, request: web.Request) -> web.Response:
        body = await request.json()
        messages = body.get("messages")
        if not isinstance(messages, list) or not messages:
            return self._bad("messages must be a non-empty list")
        sp = self._sampling(body)
        if isinstance(sp, web.Response):
            return sp
        kw = dict(body.get("chat_template_kwargs") or {})
        if body.get("tools"):
            kw["tools"] = body["tools"]
        prompt_ids = _token_ids(self.tok.apply_chat_template(messages, add_generation_prompt=True, **kw))
        req = await self.server.generate(prompt_ids, sp)
        out_ids = list(req.output_ids)
        # include_stop_str_in_output / skip_special_tokens=False (what the reference asks for): decode every id
        content = self._decode(out_ids)
        choice: dict[str, Any] = {"index": 0, "message": {"role": "assistant", "content": content, "tool_calls": []},
                                  "finish_reason": req.finish_reason, "stop_reason": None}
        if body.get("logprobs"):
            choice["logprobs"] = {"content": [{"token": f"token_id:{t}", "logprob": float(lp), "bytes": None,
                                               "top_logprobs": []} for t, lp in zip(out_ids, req.output_logprobs)]}
        else:
            choice["logprobs"] = None
        return web.json_response({
            "id": f"chatcmpl-{uuid.uuid4().hex}", "object": "chat.completion", "created": int(time.time()),
            "model": body.get("model") or self.model_name, "choices": [choice],
            "usage": {"prompt_tokens": len(prompt_ids), "completion_tokens": len(out_ids),
                      "total_tokens": len(prompt_ids) + len(out_ids)},
            "model_version": getattr(req, "model_version", None)})

    async def completions(self, request: web.Request) -> web.Response:
        body = await request.json()
        prompt = body.get("prompt")
        if int(body.get("max_tokens", 0)) != 0 or not body.get("echo"):
            return self._bad("only the scoring form is served here: max_tokens=0 with echo=true (llm.py:606-648)")
        if not isinstance(prompt, list) or not prompt:
            return self._bad("prompt must be a list of token ids or a list of such lists")
        seqs = [prompt] if isinstance(prompt[0], int) else prompt
        if any(not isinstance(s, list) or not all(isinstance(t, int) for t in s) for s in seqs):
            return self._bad("prompts must be given as token ids")
        loop = asyncio.get_running_loop()
        fut: asyncio.Future = loop.create_future()
        self._score_jobs.put((seqs, 1.0, loop, fut))     # prompt logprobs are log-softmax of the raw logits
        scored = await fut
        choices = []
        for i, (seq, lps) in enumerate(zip(seqs, scored)):
            plp: list[Any] = [None]
            for t, lp in zip(seq[1:], lps):
                plp.append({str(t): {"logprob": float(lp), "rank": None, "decoded_token": None}})
            choices.append({"index": i, "text": "", "logprobs": None, "finish_reason": "length", "prompt_logprobs": plp})
        n_tok = sum(len(s) for s in seqs)
        return web.json_response({"id": f"cmpl-{uuid.uuid4().hex}", "object": "text_completion",
                                  "created": int(time.time()), "model": body.get("model") or self.model_name,
                                  "choices": choices,
                                  "usage": {"prompt_tokens": n_tok, "completion_tokens": 0, "total_tokens": n_tok}})

    async def health(self, request: web.Request) -> web.Response:
        err = getattr(self.server, "error", None)
        if err is not None:
            return web.json_response({"status": "error", "error": repr(err)}, status=500)
        return web.Response(text="OK")

    async def receive_weight_update(self, request: web.Request) -> web.Response:
        try:
            body = await request.json()
        except Exception:  # noqa: BLE001
            body = {}
        engine = getattr(self.server, "engine", None)
        version = getattr(getattr(engine, "arena", None), "version", None)
        return web.json_response({"status": "ok", "requested_version": body.get("version"), "serving_version": version,
                                  "note": "weights arrive by the learner's P2P push; nothing to receive over HTTP"})
