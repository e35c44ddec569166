"""In-process sampler service: the thread that owns one GPU's DecodeEngine.

Replaces the vLLM API server + EngineCore + worker processes the reference launches per inference GPU
(pipelinerl/launch.py:191-247, pipelinerl/vllm1.py:189-273).  Plugins reach it through
`llm_async_generate` (async_llm.py) which submits token ids and awaits (ids, logprobs, finish_reason).
The library is not internally threaded: this single host thread drives the engine; weight-version
flips happen here, at token-step boundaries.
"""
from __future__ import annotations

import asyncio
import queue
import threading
from dataclasses import dataclass

from .engine import DecodeEngine, Request, SamplingParams

_REGISTRY: dict[str, "EngineServer"] = {}


def resolve(base_url: str) -> "EngineServer":
    if not base_url.startswith("inproc://"):
        raise ValueError(f"unsupported engine address {base_url!r} (expected inproc://<name>)")
    name = base_url[len("inproc://"):]
    if name not in _REGISTRY:
        raise KeyError(f"no sampler engine registered as {name!r}")
    return _REGISTRY[name]


def lookup(base_url: str) -> "EngineServer | None":
    """The server registered at `base_url`, or None (unsupported scheme, or nothing registered under that name)."""
    if not base_url.startswith("inproc://"):
        return None
    return _REGISTRY.get(base_url[len("inproc://"):])


@dataclass
class _Pending:
    prompt_ids: list[int]
    params: SamplingParams
    loop: asyncio.AbstractEventLoop
    future: asyncio.Future


class EngineServer:
    def __init__(self, name: str, engine: DecodeEngine, steps_per_poll: int = 4):
        self.name, self.engine = name, engine
        self.steps_per_poll = steps_per_poll
        self._inbox: "queue.Queue[_Pending]" = queue.Queue()
        self._futures: dict[int, _Pending] = {}
        self._waiting: list[_Pending] = []
        self._stop = threading.Event()
        self._thread: threading.Thread | None = None
        self.on_step_boundary = None  # callable(engine) -> None, e.g. WeightReceiver.maybe_flip
        self.tokens_generated = 0
        self.error: BaseException | None = None
        _REGISTRY[name] = self

    @property
    def base_url(self) -> str:
        return f"inproc://{self.name}"

    def start(self) -> "EngineServer":
        self._thread = threading.Thread(target=self._run, name=f"engine-{self.name}", daemon=True)
        self._thread.start()
        return self

    def stop(self) -> None:
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=30)
        _REGISTRY.pop(self.name, None)

    async def generate(self, prompt_ids: list[int], params: SamplingParams) -> Request:
        loop = asyncio.get_running_loop()
        fut: asyncio.Future = loop.create_future()
        self._inbox.put(_Pending(list(prompt_ids), params, loop, fut))
        return await fut

    # ---- engine thread ----------------------------------------------------------------------
    def _run(self) -> None:
        import torch
        eng = self.engine
        torch.cuda.set_device(eng.dev)
        try:
            while not self._stop.is_set():
                try:
                    while True:
                        self._waiting.append(self._inbox.get_nowait())
                except queue.Empty:
                    pass
                still = []
                for p in self._waiting:
                    if eng.can_admit(len(p.prompt_ids), p.params.max_tokens):
                        req = eng.add_request(p.prompt_ids, p.params, model_version=eng.arena.version)
                        self._futures[req.req_id] = p
                    else:
                        still.append(p)
                self._waiting = still
                if not eng.slot_req:
                    if self.on_step_boundary:
                        self.on_step_boundary(eng)
                    self._stop.wait(0.002)
                    continue
                for _ in range(self.steps_per_poll):
                    if self.on_step_boundary:
                        self.on_step_boundary(eng)
                    eng.step()
                for req in eng.harvest():
                    self.tokens_generated += len(req.output_ids)
                    p = self._futures.pop(req.req_id)
                    p.loop.call_soon_threadsafe(p.future.set_result, req)
        except BaseException as e:  # fail-stop: forward to every waiter (reference: actor.py:162-174)
            self.error = e
            for p in list(self._futures.values()) + self._waiting:
                p.loop.call_soon_threadsafe(p.future.set_exception, e)
            raise
