"""top-k / top-p sampling without a GPU: the oracle against vLLM 0.22's own function (tests/golden/topk_topp_cases.npz,
make_golden_topk_topp.py), request validation, both client doors and the C entry point's argument checks."""
import asyncio

import numpy as np
import pytest
import torch

from oracle.sampling_oracle import kept_mask, processed_logprobs, scaled_logits, synthetic_logits
from tests.helpers import GOLDEN, tiny_chat_tokenizer


def golden_rows():
    """(row fields, logits) of every golden row; regenerated rows are checked against their recorded checksum."""
    d = np.load(GOLDEN / "topk_topp_cases.npz")
    for i in range(len(d["V"])):
        r = {k: d[k][i] for k in d.files if k != "logits"}
        if int(r["logits_idx"]) >= 0:
            logits = torch.from_numpy(d["logits"][int(r["logits_idx"])])
        else:
            logits = synthetic_logits(str(r["kind"]), int(r["V"]), int(r["seed"]))
            assert float(logits.double().sum()) == float(r["checksum"]), "torch CPU RNG drifted: regenerate the golden"
            assert float(logits.double().abs().sum()) == float(r["checksum_abs"])
        yield r, logits


def test_oracle_reproduces_vllm_golden():
    n_rows = n_topk_only = 0
    for r, logits in golden_rows():
        V, k, p = int(r["V"]), int(r["k"]), float(r["p"])
        z = scaled_logits(logits, float(r["T"]))
        keep = kept_mask(z, k, p)
        kept = int(keep.sum())
        if p < 1.0:
            assert abs(kept - int(r["kept"])) <= int(r["band"]), (r["kind"], V, float(r["T"]), k, p, kept, int(r["kept"]))
        else:
            assert kept == int(r["kept"]), (r["kind"], V, k, kept, int(r["kept"]))   # exact, ties at the k-th value too
            n_topk_only += 1
        # 1e-6 relative (a few fp32 ulps); vLLM's own fp32 log_softmax over tens of thousands of kept tokens carries
        # ~sqrt(n) * eps of summation error (4e-5 measured at V = 152064), which the float64 oracle does not share
        lp = processed_logprobs(z, keep)[torch.from_numpy(r["ids"])].numpy()
        tol = 1e-6 * np.maximum(1.0, np.abs(r["lps"])) + (1e-4 if kept > 4096 else 0.0)
        assert (np.abs(lp - r["lps"]) <= tol).all(), (r["kind"], V, k, p, np.abs(lp - r["lps"]).max())
        n_rows += 1
    assert n_rows >= 90 and n_topk_only >= 30


def test_oracle_tie_rule_keeps_every_token_tied_with_the_boundary():
    z = torch.tensor([3.0, 2.0, 2.0, 2.0, 1.0, 0.0])
    assert kept_mask(z, 2, 1.0).tolist() == [True, True, True, True, False, False]
    # top-p boundary inside the tie: vLLM's unstable sort could split it, the contract keeps the whole tie
    w = torch.softmax(z.double(), 0)
    p = float(w[0] + w[1] + 0.5 * w[2])
    assert kept_mask(z, -1, p).tolist() == [True, True, True, True, False, False]
    assert kept_mask(z, -1, float(w[0]) * 0.5).tolist() == [True, False, False, False, False, False]


def test_sampling_params_validate_filters_as_vllm():
    from pipelinerl_b200.engine import SamplingParams
    for ok in ({"top_k": -1}, {"top_k": 0}, {"top_k": 50}, {"top_k": 10**9}, {"top_p": 1.0}, {"top_p": 1},
               {"top_p": 1e-6}, {"top_k": 50, "top_p": 0.95}):
        SamplingParams(**ok)
    for bad in ({"top_k": -2}, {"top_k": 1.5}, {"top_k": True}, {"top_k": "50"}, {"top_p": 0.0}, {"top_p": -0.1},
                {"top_p": 1.5}, {"top_p": float("nan")}, {"top_p": "0.9"}):
        with pytest.raises(ValueError):
            SamplingParams(**bad)
    V = 1000
    assert SamplingParams(top_k=50).filtered(V) and SamplingParams(top_p=0.95).filtered(V)
    assert SamplingParams(top_k=V - 1).filtered(V)
    for off in ({"top_k": -1}, {"top_k": 0}, {"top_k": V}, {"top_p": 1.0}, {"top_k": 5, "greedy": True}):
        assert not SamplingParams(**off).filtered(V)


def test_add_request_validates_filters_before_touching_the_device():
    """add_request re-checks the values (a SamplingParams may be edited after construction) before any device write;
    an engine without the filter stage rejects filtered requests."""
    from pipelinerl_b200.engine import DecodeEngine, SamplingParams
    from tests.helpers import tiny_cfg
    eng = DecodeEngine.__new__(DecodeEngine)   # host-side fields only: the checks run before any tensor is touched
    eng.cfg, eng.max_seq_len, eng.max_new, eng.fused_head = tiny_cfg("gqa2"), 64, 16, False
    params = SamplingParams(max_tokens=4)
    params.top_p = 1.5
    with pytest.raises(ValueError, match="top_p"):
        eng.add_request([1, 2, 3], params)
    params.top_p, params.top_k = 0.9, -3
    with pytest.raises(ValueError, match="top_k"):
        eng.add_request([1, 2, 3], params)
    eng.fused_head, eng._greedy, eng._temperature = True, False, 1.0
    assert not eng.supports_top_k_top_p
    with pytest.raises(ValueError, match="top-k / top-p"):
        eng.add_request([1, 2, 3], SamplingParams(max_tokens=4, top_k=50, top_p=0.95))
    from pipelinerl_b200.tp_engine import TPDecodeEngine
    tp = TPDecodeEngine.__new__(TPDecodeEngine)
    tp.cfg, tp.max_seq_len, tp.max_new, tp.fused_head = tiny_cfg("gqa2"), 64, 16, False
    assert not tp.supports_top_k_top_p
    for filt in ({"top_k": 50}, {"top_p": 0.95}):
        with pytest.raises(ValueError, match="top-k / top-p"):
            tp.add_request([1, 2, 3], SamplingParams(max_tokens=4, **filt))


class _CapableEngine:
    supports_top_k_top_p = True


class _RecordingServer:
    def __init__(self, engine):
        self.engine, self.params, self.on_step_boundary, self.error = engine, [], None, None

    async def generate(self, prompt_ids, params):
        import types
        self.params.append(params)
        return types.SimpleNamespace(output_ids=[3, 4], output_logprobs=[-0.5, -0.25], finish_reason="length",
                                     model_version=0)


def test_in_process_door_passes_filters_to_capable_engines_only():
    from pipelinerl_b200 import serving
    from pipelinerl_b200.async_llm import llm_async_generate
    from pipelinerl_b200.llm import Prompt, SyntheticTokenizer, TrainableLLM
    prompt = Prompt(messages=[{"role": "user", "content": "hi"}])
    params = {"max_tokens": 2, "temperature": 1.0, "top_p": 0.95, "top_k": 50}
    capable = _RecordingServer(_CapableEngine())
    serving._REGISTRY["filters-ok"] = capable
    serving._REGISTRY["filters-no"] = _RecordingServer(object())
    try:
        llm = TrainableLLM("inproc://filters-ok", "m", parameters=params, tokenizer=SyntheticTokenizer())
        call = asyncio.run(llm_async_generate(llm, prompt))
        assert call.output_length_tokens == 2
        sp = capable.params[-1]
        assert (sp.top_k, sp.top_p, sp.temperature, sp.greedy) == (50, 0.95, 1.0, False)
        for bad in ({"top_p": 1.5}, {"top_k": -2}, {"top_p": 0.0}):
            llm = TrainableLLM("inproc://filters-ok", "m", parameters={**params, **bad}, tokenizer=SyntheticTokenizer())
            with pytest.raises(ValueError):
                asyncio.run(llm_async_generate(llm, prompt))
        for url in ("inproc://filters-no", "inproc://nobody-here", "http://elsewhere:8000"):
            llm = TrainableLLM(url, "m", parameters=params, tokenizer=SyntheticTokenizer())
            with pytest.raises(ValueError):
                asyncio.run(llm_async_generate(llm, prompt))
        assert serving.lookup("inproc://nobody-here") is None and serving.lookup("http://x") is None
        assert serving.lookup("inproc://filters-ok") is capable
    finally:
        serving._REGISTRY.pop("filters-ok", None)
        serving._REGISTRY.pop("filters-no", None)


def test_http_door_accepts_filters_on_capable_engines():
    import aiohttp
    from pipelinerl_b200.http_shim import HttpShim
    from tests.test_http_shim import FakeServer

    async def go():
        server = FakeServer().start()
        server.engine.supports_top_k_top_p = True
        seen = []
        inner = server.generate

        async def generate(prompt_ids, params):
            seen.append(params)
            return await inner(prompt_ids, params)
        server.generate = generate
        shim = HttpShim(server, tiny_chat_tokenizer(), "tiny")
        url = await shim.start()
        msg = {"model": "tiny", "messages": [{"role": "user", "content": "hello"}], "logprobs": True}
        try:
            async with aiohttp.ClientSession() as s:
                async with s.post(url + "/v1/chat/completions", json={**msg, "top_p": 0.95, "top_k": 50}) as r:
                    assert r.status == 200
                    assert len((await r.json())["choices"][0]["logprobs"]["content"]) > 0
                assert (seen[-1].top_k, seen[-1].top_p) == (50, 0.95)
                async with s.post(url + "/v1/chat/completions", json={**msg, "top_p": None, "top_k": None}) as r:
                    assert r.status == 200
                assert (seen[-1].top_k, seen[-1].top_p) == (-1, 1.0)
                n_ok = len(seen)
                for bad in ({"top_p": 0}, {"top_p": 1.5}, {"top_k": -2}, {"top_k": 2.5}):
                    async with s.post(url + "/v1/chat/completions", json={**msg, **bad}) as r:
                        assert r.status == 400 and "error" in await r.json(), bad
                assert len(seen) == n_ok
                server.engine.supports_top_k_top_p = False
                for bad in ({"top_p": 0.9}, {"top_k": 20}, {"top_p": 1.5}):
                    async with s.post(url + "/v1/chat/completions", json={**msg, **bad}) as r:
                        assert r.status == 400, bad
        finally:
            await shim.stop()
            server.stop()
    asyncio.new_event_loop().run_until_complete(go())


def test_filter_entry_point_validates_arguments_without_a_gpu():
    from pipelinerl_b200 import _build, _lib
    _build.build(verbose=False)
    lib, P = _lib.load(), 0x1000
    assert lib.prl_sample_filter_workspace_bytes(64, 152064) == 0
    cases = [
        (lambda: lib.prl_sample_filter_rows(None, 4, 100, P, P, P, P, 0, 0, P, P, None, None, 0, None), b"NULL"),
        (lambda: lib.prl_sample_filter_rows(P, 4, 100, P, P, None, P, 0, 0, P, P, None, None, 0, None), b"NULL"),
        (lambda: lib.prl_sample_filter_rows(P, 4, 100, P, P, P, P, 0, 0, P, None, None, None, 0, None), b"NULL"),
        (lambda: lib.prl_sample_filter_rows(P, 0, 100, P, P, P, P, 0, 0, P, P, None, None, 0, None), b"bad shape"),
        (lambda: lib.prl_sample_filter_rows(P, 4, 0, P, P, P, P, 0, 0, P, P, None, None, 0, None), b"bad shape"),
        (lambda: lib.prl_sample_filter_rows(P, 4, 1 << 24, P, P, P, P, 0, 0, P, P, None, None, 0, None), b"exceeds"),
        (lambda: lib.prl_sample_filter_rows(P, 4, 100, P, P, P, P, 0, 0, P, P, None, None, 64, None), b"workspace"),
    ]
    for call, needle in cases:
        assert call() < 0
        assert needle in lib.prl_last_error(), (needle, lib.prl_last_error())
