"""Client side of the plugin surface: `llm_async_generate` and `make_training_text`
(reference: pipelinerl/async_llm.py:86-212 and :215-346)."""
from __future__ import annotations

from .engine import SamplingParams
from .llm import LLMCall, LLMOutput, Prompt, TokenLogprob, TrainableLLM
from .rollouts import TrainingText, apply_rollout_reward
from .serving import lookup, resolve

MASKED_TOKEN_ID = -100


class RetryableAbortedCompletionError(TimeoutError):
    """Abort-shaped completion that should be retried instead of treated as data."""


def _field(obj, name):
    """tool calls arrive as pydantic objects (litellm types in the reference) or as plain dicts"""
    return obj[name] if isinstance(obj, dict) else getattr(obj, name)


def _token_ids(encoded) -> list[int]:
    """apply_chat_template(tokenize=True) returns a list of ids with the transformers the reference pins (4.57) and a
    BatchEncoding with transformers >= 5: accept both."""
    if hasattr(encoded, "keys") and "input_ids" in encoded.keys():
        encoded = encoded["input_ids"]
    return list(encoded)


def _chat_kwargs(llm: TrainableLLM, prompt: Prompt) -> dict:
    kw = dict(llm.chat_template_kwargs or {})
    if prompt.tools:
        kw["tools"] = prompt.tools
    return kw


def _filters_supported(base_url: str) -> bool:
    """Whether the engine behind `base_url` samples with top-k / top-p (DecodeEngine without the fused head)."""
    server = lookup(base_url)
    return bool(getattr(getattr(server, "engine", None), "supports_top_k_top_p", False))


def _reject_unsupported_sampling(params: dict, filters_supported: bool) -> None:
    """Sampling features the engine does not implement must fail loudly, exactly as http_shim.py answers 400 for them:
    a silently ignored top_p / top_k / stop would make the recorded logprobs those of a different distribution than the
    one the request asked for.  (The reference trains with top_p = 1, top_k = -1, no stop strings: conf/base.yaml:46-51;
    its eval handle samples with top_p 0.95, top_k 50, which engines with `supports_top_k_top_p` serve.)"""
    if not filters_supported and (float(params.get("top_p") or 1.0) < 1.0 or int(params.get("top_k") or -1) > 0):
        raise ValueError("top_p / top_k sampling is not implemented by this engine")
    if params.get("stop") or params.get("stop_token_ids"):
        raise ValueError("stop strings / stop token ids are not implemented by this engine (eos only)")
    if int(params.get("n", 1)) != 1:
        raise ValueError("n > 1 completions per request is not implemented (the actor issues `attempts` requests)")
    for name in ("presence_penalty", "frequency_penalty", "repetition_penalty", "min_p"):
        if params.get(name) not in (None, 0, 0.0, 1, 1.0) or (name == "repetition_penalty" and params.get(name) not in (None, 1, 1.0)):
            raise ValueError(f"sampling parameter {name} is not implemented by this engine")


async def llm_async_generate(llm: TrainableLLM, prompt: Prompt, session=None,
                             max_tokens_override: int | None = None) -> LLMCall:
    """One completion.  `session` (an aiohttp.ClientSession in the reference) is accepted and unused: the
    engine is in-process.  Returns an LLMCall with .output.content, .logprobs[i].{token_id, logprob},
    .prompt_length_tokens, .output_length_tokens and .llm_info['finish_reason'] in {stop, length}."""
    tok = llm.load_tokenizer()
    prompt_ids = prompt.token_ids or _token_ids(tok.apply_chat_template(prompt.messages, add_generation_prompt=True,
                                                                        **_chat_kwargs(llm, prompt)))
    params = llm.parameters
    _reject_unsupported_sampling(params, _filters_supported(llm.base_url))
    max_tokens = int(max_tokens_override if max_tokens_override is not None else params.get("max_tokens", 16))
    temperature = float(params.get("temperature", 1.0))
    sp = SamplingParams(max_tokens=max_tokens, temperature=temperature if temperature > 0 else 1.0,
                        greedy=temperature <= 0, ignore_eos=bool(params.get("ignore_eos", False)),
                        top_k=-1 if params.get("top_k") is None else params["top_k"],
                        top_p=1.0 if params.get("top_p") is None else params["top_p"])
    req = await resolve(llm.base_url).generate(list(prompt_ids), sp)
    content = tok.decode(req.output_ids)
    call = llm.log_output(prompt, LLMOutput(content=content), count_tokens=False)
    call.prompt_length_tokens = len(prompt_ids)
    call.output_length_tokens = len(req.output_ids)
    call.llm_info["finish_reason"] = req.finish_reason
    call.llm_info["model_version"] = req.model_version
    call.llm_info["prompt_token_ids"] = list(prompt_ids)
    if llm.collect_logprobs:
        call.logprobs = [TokenLogprob(token_id=t, logprob=lp) for t, lp in zip(req.output_ids, req.output_logprobs)]
    return call


def make_training_text(llm: TrainableLLM, llm_call: LLMCall) -> TrainingText:
    """input_ids = prompt ids + generated ids; labels mask the prompt; logprobs are the sampler's."""
    finish_reason = llm_call.llm_info.get("finish_reason")
    if finish_reason == "abort":
        raise RetryableAbortedCompletionError(f"Aborted completion for prompt {llm_call.prompt.id} should be retried")
    if not llm_call.logprobs:
        raise ValueError("Logprobs are required to make training data for RL")
    tok = llm.load_tokenizer()
    kw = _chat_kwargs(llm, llm_call.prompt)
    prompt_ids = llm_call.llm_info.get("prompt_token_ids")
    if prompt_ids is None:
        prompt_ids = _token_ids(tok.apply_chat_template(llm_call.prompt.messages, add_generation_prompt=True, **kw))
    prompt_text = tok.apply_chat_template(llm_call.prompt.messages, tokenize=False, add_generation_prompt=True, **kw)
    assistant: dict = {"role": "assistant", "content": llm_call.output.content or ""}
    if llm_call.output.tool_calls:   # rendered by the chat template exactly as the reference passes them (:227-238)
        assistant["tool_calls"] = [{"id": _field(tc, "id"), "type": "function",
                                    "function": {"name": _field(_field(tc, "function"), "name"),
                                                 "arguments": _field(_field(tc, "function"), "arguments")}}
                                   for tc in llm_call.output.tool_calls]
    full = llm_call.prompt.messages + [assistant]
    text = tok.apply_chat_template(full, tokenize=False, **kw)
    output_text = text[len(prompt_text):]
    bos = getattr(tok, "bos_token", None)
    if bos and text.startswith(bos):
        text = text[len(bos):]
    gen = [lp.token_id for lp in llm_call.logprobs]
    if finish_reason is not None:
        finished = finish_reason != "length"
    else:
        eos = getattr(tok, "eos_token", "") or ""
        finished = bool(eos) and (llm_call.output.content or "").endswith(eos)
    return TrainingText(text=text, n_predicted=len(output_text), input_ids=list(prompt_ids) + gen,
                        labels=[MASKED_TOKEN_ID] * len(prompt_ids) + gen,
                        logprobs=[lp.logprob for lp in llm_call.logprobs], finished=finished,
                        prompt_tokens=llm_call.prompt_length_tokens, output_tokens=llm_call.output_length_tokens)


def make_training_texts_from_llm_calls(llm: TrainableLLM, llm_calls: list[LLMCall], reward: float | None = None):
    texts = [make_training_text(llm, c) for c in llm_calls]
    return apply_rollout_reward(texts, reward) if reward is not None else texts
