"""top-k / top-p sampling on the GPU: prl_sample_filter_rows against vLLM 0.22's own function
(tests/golden/topk_topp_cases.npz), its invariants (untouched rows, shared Gumbel noise, the filtered distribution), and
the engine serving filtered and unfiltered requests in one batch."""
import asyncio

import numpy as np
import pytest
import torch

from oracle.sampling_oracle import kept_mask, processed_logprobs, scaled_logits
from tests.helpers import tiny_cfg, tiny_weights
from tests.test_sampling_filters import golden_rows

pytestmark = pytest.mark.gpu


class Sampler:
    """prl_sample_logprob_rows followed by prl_sample_filter_rows on [B, V] logits, as the engine runs them."""

    def __init__(self, logits, temps, top_k, top_p, greedy=None):
        from pipelinerl_b200 import _lib
        self.lib, self._lib = _lib.load(), _lib
        dev = logits.device
        self.B, self.V = logits.shape
        self.logits = logits.contiguous()
        self.inv_t = torch.tensor([1.0 / t for t in temps], dtype=torch.float32, device=dev)
        self.greedy = torch.tensor(greedy if greedy is not None else [0] * self.B, dtype=torch.uint8, device=dev)
        self.top_k = torch.tensor(top_k, dtype=torch.int32, device=dev)
        self.top_p = torch.tensor(top_p, dtype=torch.float32, device=dev)
        self.ws = torch.zeros(int(self.lib.prl_sample_workspace_bytes(self.B)), dtype=torch.uint8, device=dev)
        self.ids = torch.zeros(self.B, dtype=torch.int32, device=dev)
        self.lps = torch.zeros(self.B, dtype=torch.float32, device=dev)
        self.kept = torch.zeros(self.B, dtype=torch.int32, device=dev)

    def unfiltered(self, step, seed=1234):
        self._lib.check(self.lib.prl_sample_logprob_rows(self.logits.data_ptr(), self.B, self.V, self.inv_t.data_ptr(),
                                                         self.greedy.data_ptr(), seed, step, self.ids.data_ptr(),
                                                         self.lps.data_ptr(), self.ws.data_ptr(), self.ws.numel(), None))
        return self.ids.clone(), self.lps.clone()

    def filtered(self, step, seed=1234):
        self.unfiltered(step, seed)
        self._lib.check(self.lib.prl_sample_filter_rows(self.logits.data_ptr(), self.B, self.V, self.inv_t.data_ptr(),
                                                        self.greedy.data_ptr(), self.top_k.data_ptr(),
                                                        self.top_p.data_ptr(), seed, step, self.ids.data_ptr(),
                                                        self.lps.data_ptr(), self.kept.data_ptr(), None, 0, None))
        return self.ids.clone(), self.lps.clone(), self.kept.clone()


def test_filter_kernel_matches_vllm_golden(cuda_device):
    groups: dict[int, list] = {}
    for r, logits in golden_rows():
        groups.setdefault(int(r["V"]), []).append((r, logits))
    n_checked = 0
    for V, rows in groups.items():
        logits = torch.stack([lg for _, lg in rows]).to(cuda_device)
        s = Sampler(logits, [float(r["T"]) for r, _ in rows], [int(r["k"]) for r, _ in rows],
                    [float(r["p"]) for r, _ in rows])
        z = torch.stack([scaled_logits(lg, float(r["T"])) for r, lg in rows])
        first = None
        for step in range(4):
            ids, lps, kept = (t.cpu() for t in s.filtered(step))
            if first is None:
                first = (ids, lps, kept)
            for b, (r, _) in enumerate(rows):
                k, p, i = int(r["k"]), float(r["p"]), int(ids[b])
                if p < 1.0:
                    assert abs(int(kept[b]) - int(r["kept"])) <= int(r["band"]), (V, b, int(kept[b]), int(r["kept"]))
                else:
                    assert int(kept[b]) == int(r["kept"]), (V, b, int(kept[b]), int(r["kept"]))
                assert float(z[b, i]) >= float(r["min_kept_z"]), (V, b, i)          # inside vLLM's kept set
                want = float(z[b, i]) - float(r["lse"])
                assert abs(float(lps[b]) - want) <= 1e-4, (V, b, k, p, float(lps[b]), want)
                n_checked += 1
        again = s.filtered(0)   # deterministic: the same inputs give the same bits
        assert all(torch.equal(a.cpu(), f) for a, f in zip(again, first))
    assert n_checked >= 4 * 90


def test_unfiltered_and_greedy_rows_are_left_untouched(cuda_device):
    g = torch.Generator().manual_seed(5)
    B, V = 8, 152064
    logits = (torch.randn(B, V, generator=g) * 2).to(cuda_device)
    #          off     k=V     p=1,k=0   greedy+filters     filtered rows
    top_k = [-1, V, 0, 50, 50, -1, 50, 7]
    top_p = [1.0, 1.0, 1.0, 0.9, 0.95, 0.5, 1.0, 0.3]
    greedy = [0, 0, 0, 1, 0, 0, 0, 0]
    s = Sampler(logits, [1.0, 0.7, 1.3, 1.0, 1.0, 0.8, 1.0, 1.0], top_k, top_p, greedy)
    for step in range(3):
        ids0, lps0 = s.unfiltered(step)
        ids, lps, kept = s.filtered(step)
        for b in (0, 1, 2, 3):
            assert torch.equal(ids[b], ids0[b]) and torch.equal(lps[b], lps0[b]), b
            assert int(kept[b]) == V
        assert (kept[4:] < V).all()


def test_filtered_sample_shares_the_unfiltered_noise(cuda_device):
    """Same counter-based Gumbel noise: whenever the unfiltered sample lies in the kept set, the filtered one equals it."""
    g = torch.Generator().manual_seed(9)
    B, V = 64, 4096
    base = torch.randn(B, V, generator=g) * torch.linspace(0.5, 3.0, B)[:, None]
    configs = [(50, 0.95), (-1, 0.9), (20, 1.0), (-1, 0.5)] * (B // 4)
    temps = [0.7, 1.0, 1.3, 1.0] * (B // 4)
    s = Sampler(base.to(cuda_device), temps, [k for k, _ in configs], [p for _, p in configs])
    masks = torch.stack([kept_mask(scaled_logits(base[b], temps[b]), *configs[b]) for b in range(B)])
    same = 0
    for step in range(50):
        ids0, _ = s.unfiltered(step)
        ids, _, kept = s.filtered(step)
        ids0, ids = ids0.cpu().long(), ids.cpu().long()
        assert masks[torch.arange(B), ids].all()
        inside = masks[torch.arange(B), ids0]
        assert torch.equal(ids[inside], ids0[inside])
        same += int(inside.sum())
    assert same >= 500


def test_filtered_sampling_distribution(cuda_device):
    """25 600 draws of one V = 1000 row at T = 0.8, k = 50, p = 0.9: none outside the kept set, and the 20 most likely
    kept ids within 5 sigma of their renormalised expectation."""
    B, V, T = 64, 1000, 0.8
    g = torch.Generator().manual_seed(0)
    row = torch.randn(V, generator=g) * 2
    s = Sampler(row.repeat(B, 1).to(cuda_device), [T] * B, [50] * B, [0.9] * B)
    z = scaled_logits(row, T)
    keep = kept_mask(z, 50, 0.9)
    ref = processed_logprobs(z, keep)
    counts = torch.zeros(V)
    for step in range(400):
        ids, lps, kept = s.filtered(step)
        i = ids.cpu().long()
        assert torch.allclose(lps.cpu(), ref[i], atol=1e-4)
        assert (kept.cpu() == int(keep.sum())).all()
        counts += torch.bincount(i, minlength=V).float()
    n = counts.sum()
    assert counts[~keep].sum() == 0
    p = ref.exp()
    top = torch.topk(p, 20).indices
    sigma = torch.sqrt(n * p[top] * (1 - p[top]))
    assert ((counts[top] - n * p[top]).abs() < 5 * sigma + 1).all()


def _engine(kind, dev, **kw):
    from pipelinerl_b200.engine import DecodeEngine
    from pipelinerl_b200.model import ParamArena
    cfg = tiny_cfg(kind)
    w = tiny_weights(cfg)
    arena = ParamArena(cfg, dev)
    for name in arena.names():
        arena.view(name).copy_(w[name].to(torch.bfloat16))
    return cfg, DecodeEngine(cfg, arena, device=dev, **kw)


@pytest.mark.parametrize("kind,use_graph", [("gqa2", True), ("gqa2", False), ("gqa7", True), ("gqa7", False)])
def test_engine_mixed_batch(cuda_device, kind, use_graph):
    from pipelinerl_b200.engine import SamplingParams
    mk = dict(max_batch=4, max_seq_len=128, max_new_tokens=16, use_cuda_graph=use_graph, prefill_chunk=0)
    cfg, eng = _engine(kind, cuda_device, **mk)
    g = torch.Generator().manual_seed(3)
    prompt = torch.randint(0, cfg.vocab_size, (9,), generator=g).tolist()
    plain = SamplingParams(max_tokens=8, temperature=1.0)
    params = [plain, SamplingParams(max_tokens=8, temperature=1.0, top_k=50, top_p=0.95),
              SamplingParams(max_tokens=8, temperature=0.7, top_p=0.8),
              SamplingParams(max_tokens=8, greedy=True, top_k=5)]
    reqs = [eng.add_request(prompt, p) for p in params]      # the unfiltered request first: same slot in both runs
    assert eng._n_filtered == 2
    checked = 0
    for _ in range(len(prompt) + 8):
        eng.step()
        logits, ids, lps = eng.logits.cpu(), eng.sampled.cpu(), eng.sampled_lp.cpu()
        for r, p in zip(reqs, params):
            sl = r.slot
            if p.greedy:
                z, keep = logits[sl], torch.ones(cfg.vocab_size, dtype=torch.bool)
                assert int(ids[sl]) == int(torch.argmax(z))
            else:
                z = scaled_logits(logits[sl], p.temperature)
                keep = kept_mask(z, p.top_k, p.top_p)
            assert bool(keep[int(ids[sl])]), (sl, int(ids[sl]))
            ref = processed_logprobs(z, keep)
            assert abs(float(lps[sl]) - float(ref[int(ids[sl])])) <= 2e-4, (sl, float(lps[sl]), float(ref[int(ids[sl])]))
            checked += 1
    assert checked == 4 * (len(prompt) + 8)
    done = {r.req_id: r for r in eng.harvest()}
    assert len(done) == 4 and eng._n_filtered == 0
    assert (eng.top_k_rows.cpu() == -1).all() and (eng.top_p_rows.cpu() == 1.0).all()
    # the unfiltered request alone: bit-identical ids and logprobs
    _, solo = _engine(kind, cuda_device, **mk)
    r0 = solo.add_request(prompt, plain)
    for _ in range(len(prompt) + 8):
        solo.step()
    alone = {r.req_id: r for r in solo.harvest()}[r0.req_id]
    mixed = done[reqs[0].req_id]
    assert alone.output_ids == mixed.output_ids
    assert np.array_equal(np.array(alone.output_logprobs, dtype=np.float32), np.array(mixed.output_logprobs, dtype=np.float32))


def test_engines_without_a_filter_stage_reject_filtered_requests(cuda_device):
    from pipelinerl_b200.engine import SamplingParams
    _, eng = _engine("gqa2", cuda_device, max_batch=2, max_seq_len=64, max_new_tokens=8, fused_head=True)
    assert not eng.supports_top_k_top_p
    with pytest.raises(ValueError):
        eng.add_request([1, 2, 3], SamplingParams(max_tokens=4, top_k=50, top_p=0.95))
    eng.add_request([1, 2, 3], SamplingParams(max_tokens=4, top_k=-1, top_p=1.0))   # unfiltered: still served
    # TPDecodeEngine (2 GPUs, one process per rank) takes the same add_request path: tests/test_sampling_filters.py


def test_plugin_door_serves_the_eval_handle(cuda_device):
    """llm_async_generate with the reference's eval-handle parameters through a real EngineServer: every filtered
    logprob is >= the unfiltered teacher-forced logprob of the same token (renormalising over a subset only raises it),
    less the end-to-end bf16 bound."""
    from pipelinerl_b200.async_llm import llm_async_generate
    from pipelinerl_b200.llm import Prompt, SyntheticTokenizer, TrainableLLM
    from pipelinerl_b200.serving import EngineServer
    cfg, eng = _engine("gqa2", cuda_device, max_batch=4, max_seq_len=192, max_new_tokens=32)
    assert eng.supports_top_k_top_p
    server = EngineServer("filter-eval", eng).start()
    try:
        tok = SyntheticTokenizer(vocab_size=cfg.vocab_size)
        llm = TrainableLLM(server.base_url, "tiny", tokenizer=tok,
                           parameters={"max_tokens": 16, "temperature": 1.0, "top_p": 0.95, "top_k": 50})

        async def run():
            prompts = [Prompt(messages=[{"role": "user", "content": f"count {i} 7 11 13"}]) for i in range(3)]
            return await asyncio.gather(*(llm_async_generate(llm, pr) for pr in prompts))
        calls = asyncio.run(run())
    finally:
        server.stop()
    for call in calls:
        assert call.output_length_tokens == 16 and len(call.logprobs) == 16
        seq = call.llm_info["prompt_token_ids"] + [lp.token_id for lp in call.logprobs]
        teacher = eng.score([seq])[0][-16:]
        for lp, t in zip(call.logprobs, teacher):
            assert lp.logprob <= 1e-6 and lp.logprob >= t - 3e-2, (lp.logprob, t)
