"""Sampler engine: continuous-batching token-step loop on one GPU, over libprl.so.

This is what replaces the vLLM server of the reference for hot path 1 (launch:
pipelinerl/launch.py:191-247; per-request client: pipelinerl/async_llm.py:86-212).  One engine
owns one GPU: a parameter arena (model.ParamArena), a paged KV pool, device-resident per-slot
scheduler state, and a CUDA graph of the whole token step (all ~290 kernel launches of a 28-layer
model replayed with one call).  The host only admits requests into free slots and harvests
finished ones; token feeding, sampling, logprob capture and retirement happen on the device
(prl_advance_state), so there is no per-token host round trip.

Requests carry token ids in and (token ids, logprobs, finish_reason) out — the fields
`make_training_text` needs (async_llm.py:215-346).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field

import torch

from . import _lib
from .model import ModelConfig, ParamArena

PAGE_SIZE = 64


@dataclass
class SamplingParams:
    max_tokens: int = 16
    temperature: float = 1.0
    greedy: bool = False
    ignore_eos: bool = False
    # vLLM's filters (the reference's eval handle: top_p 0.95, top_k 50): top_k in {-1, 0} or >= vocabulary and
    # top_p == 1 disable them; greedy requests ignore both.  Logprobs are then those of the filtered, renormalised
    # distribution (processed_logprobs).
    top_k: int = -1
    top_p: float = 1.0

    def __post_init__(self):
        self.check_filters()

    def check_filters(self) -> None:
        """The values vLLM accepts (sampling_params.py:_verify_args): top_k an integer >= -1, top_p in (0, 1]."""
        if isinstance(self.top_k, bool) or not isinstance(self.top_k, int) or self.top_k < -1:
            raise ValueError(f"top_k must be an integer >= -1 (-1 or 0 disables it), got {self.top_k!r}")
        if isinstance(self.top_p, bool) or not isinstance(self.top_p, (int, float)) or not 0.0 < self.top_p <= 1.0:
            raise ValueError(f"top_p must be in (0, 1], got {self.top_p!r}")

    def filtered(self, vocab_size: int) -> bool:
        """True when top-k or top-p changes this request's distribution."""
        return not self.greedy and (1 <= self.top_k < vocab_size or self.top_p < 1.0)


@dataclass
class Request:
    req_id: int
    prompt_ids: list[int]
    params: SamplingParams
    slot: int = -1
    pages: list[int] = field(default_factory=list)
    output_ids: list[int] = field(default_factory=list)
    output_logprobs: list[float] = field(default_factory=list)
    finish_reason: str | None = None
    model_version: int = 0
    prefilled: int = 0                                   # prompt tokens whose KV is in the cache
    waits_for: list = field(default_factory=list)        # [(request filling a shared page, tokens it must reach)]
    filtered: bool = False                               # holds its slot's top-k / top-p rows


class DecodeEngine:
    def __init__(self, cfg: ModelConfig, arena: ParamArena, max_batch: int = 64, max_seq_len: int = 16384,
                 n_pages: int | None = None, max_new_tokens: int = 8192, eos_id: int = -1, seed: int = 42,
                 device: torch.device | str = "cuda:0", use_cuda_graph: bool = True, prefill_chunk: int = 1024,
                 prefix_sharing: bool = True, fused_head: bool = False):
        if cfg.head_dim != 128:
            raise ValueError("the sm_100a attention kernel is built for head_dim 128")
        self.cfg, self.arena = cfg, arena
        self.lib = _lib.load()
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise RuntimeError("DecodeEngine needs a CUDA device: pipelinerl_b200 has no CPU fallback")
        self.B = max_batch
        self.max_seq_len = max_seq_len
        self.max_blocks = (max_seq_len + PAGE_SIZE - 1) // PAGE_SIZE
        # page 0 is a scratch page: idle slots point at it, so their (discarded) KV writes are harmless
        self.n_pages = n_pages if n_pages is not None else 1 + self.B * self.max_blocks
        self.max_new = max_new_tokens
        self.eos_id, self.seed = eos_id, seed
        self.use_graph = use_cuda_graph
        # fused_head: lm_head + sampling + logprob capture in one GEMM epilogue (no logits in HBM).  For the 64-row
        # decode step the logits round trip is only 78 MB and the fused epilogue cannot live in the step's CUDA graph
        # (its RNG arguments change per step), so the unfused path measured 1.5 % faster (profiles/r1_ablation_b.jsonl);
        # the fused kernel is what scoring / the trainer's forward use, where the logits would be 608 KB per token.
        self.fused_head = fused_head
        self.l2_prefetch_bytes = 0          # cross-kernel L2 prefetch budget per site; measured to HURT (+0.19 ms/step,
                                            # profiles/r1_ablation.jsonl: HBM is already saturated), so off
        self._skip: set[str] = set()        # timing ablations only (tools/step_ablation.py)
        # SiLU(gate) * up in the gate_up GEMM's epilogue (prl_gemm_swiglu_decode); PRL_FUSE_SWIGLU=0 keeps the two-kernel pair
        self.fuse_swiglu = os.environ.get("PRL_FUSE_SWIGLU", "1") != "0"
        d, B, H, I = self.dev, self.B, cfg.hidden_size, cfg.intermediate_size
        kv_elems = cfg.num_layers * 2 * self.n_pages * cfg.num_kv_heads * PAGE_SIZE * cfg.head_dim
        self.kv_cache = torch.zeros(kv_elems, dtype=torch.bfloat16, device=d)
        i32 = dict(dtype=torch.int32, device=d)
        self.block_table = torch.zeros(B, self.max_blocks, **i32)
        self.tokens = torch.zeros(B, **i32)
        self.positions = torch.zeros(B, **i32)
        self.seq_lens = torch.zeros(B, **i32)
        self.active = torch.zeros(B, dtype=torch.uint8, device=d)
        self.finished = torch.zeros(B, dtype=torch.uint8, device=d)
        self.prompt_stride = max_seq_len
        self.prompt_buf = torch.zeros(B, self.prompt_stride, **i32)
        self.prompt_len = torch.zeros(B, **i32)
        self.out_ids = torch.zeros(B, self.max_new, **i32)
        self.out_logprobs = torch.zeros(B, self.max_new, dtype=torch.float32, device=d)
        self.gen_count = torch.zeros(B, **i32)
        self.max_new_t = torch.zeros(B, **i32)
        self.sampled = torch.zeros(B, **i32)
        self.sampled_lp = torch.zeros(B, dtype=torch.float32, device=d)
        # activations
        self.h = torch.zeros(B, H, dtype=torch.float32, device=d)
        self.x = torch.zeros(B, H, dtype=torch.bfloat16, device=d)
        self.q = torch.zeros(B, cfg.q_size, dtype=torch.bfloat16, device=d)
        self.attn_out = torch.zeros(B, cfg.q_size, dtype=torch.bfloat16, device=d)
        self.act = torch.zeros(B, I, dtype=torch.bfloat16, device=d)
        self.logits = torch.zeros(B, cfg.head_rows, dtype=torch.float32, device=d)
        # HF rotary: inv_freq = 1 / theta^(arange(0, d, 2) / d) in fp32
        self.inv_freq = (1.0 / (cfg.rope_theta ** (torch.arange(0, cfg.head_dim, 2, dtype=torch.int64).float()
                                                   / cfg.head_dim))).to(d)
        self._plan_gemms()
        self.attn_splits = int(self.lib.prl_paged_attn_splits(B, cfg.num_kv_heads, max_seq_len))
        self.attn_ws = torch.zeros(int(self.lib.prl_paged_attn_workspace_bytes(B, cfg.num_q_heads, self.attn_splits)),
                                   dtype=torch.uint8, device=d)
        self.sample_ws = torch.zeros(int(self.lib.prl_sample_workspace_bytes(B)), dtype=torch.uint8, device=d)
        self.head_ws = torch.zeros(int(self.lib.prl_head_workspace_bytes(B, cfg.vocab_size)), dtype=torch.uint8, device=d)
        self.free_pages = list(range(self.n_pages - 1, 0, -1))
        self.free_slots = list(range(B - 1, -1, -1))
        self.slot_req: dict[int, Request] = {}
        self.step_count = 0
        # sampling parameters are PER SLOT (device arrays read by the sampler / state-advance kernels): requests of
        # different LLM handles (train T=1, eval greedy, ...) share the batch without touching each other's distribution.
        # The engine-wide attributes below are the defaults of idle slots and what benches / tools set for all slots.
        self.inv_temp_rows = torch.ones(B, dtype=torch.float32, device=d)
        self.greedy_rows = torch.zeros(B, dtype=torch.uint8, device=d)
        self.ignore_eos_rows = torch.zeros(B, dtype=torch.uint8, device=d)
        # top-k / top-p per slot (-1 / 1.0: off).  The filter kernel runs only while some slot holds a filtered request,
        # so a batch without one launches exactly the kernels it did before the filters existed.
        self.top_k_rows = torch.full((B,), -1, dtype=torch.int32, device=d)
        self.top_p_rows = torch.ones(B, dtype=torch.float32, device=d)
        self._n_filtered = 0
        self._temperature, self._greedy, self._ignore_eos = 1.0, False, False
        self._graphs: dict[int, torch.cuda.CUDAGraph] = {}
        # ---- chunked prefill + prefix sharing (GRPO attempts share their prompt) ----
        self.prefill_chunk = int(prefill_chunk)
        self.prefill_attn_tc = os.environ.get("PRL_PREFILL_ATTN", "tc") != "mma"   # tcgen05 (default) | mma.sync kernel
        self.prefix_sharing = prefix_sharing
        self.page_ref = [0] * self.n_pages
        self._prefill_queue: list[Request] = []
        from collections import OrderedDict
        self._page_of_hash: "OrderedDict[int, int]" = OrderedDict()   # chained hash of a full 64-token page -> page id (LRU)
        self._hash_of_page: dict[int, int] = {}
        self._tokens_of_page: dict[int, tuple] = {}                   # page -> its 64 tokens (verified on every hit)
        self._page_pending: dict[int, tuple[Request, int]] = {}       # page -> (request that fills it, tokens needed)
        self._pf = None                                # lazily allocated prefill buffers
        self.stats = {"prefill_tokens": 0, "prefix_hits": 0, "prefix_hit_tokens": 0}
        self.profile_timing = False                    # benches: wall time spent inside run_prefill (costs two syncs per call)
        self._next_id = 0
        self._state = self._make_state()

    # engine-wide sampling defaults: assigning one overwrites every slot (benches, tools, single-tenant tests)
    @property
    def temperature(self) -> float:
        return self._temperature

    @temperature.setter
    def temperature(self, t: float) -> None:
        if not t > 0:
            raise ValueError("temperature must be > 0 (use greedy=True for argmax)")
        self._temperature = float(t)
        self.inv_temp_rows.fill_(1.0 / float(t))

    @property
    def greedy(self) -> bool:
        return self._greedy

    @greedy.setter
    def greedy(self, g: bool) -> None:
        self._greedy = bool(g)
        self.greedy_rows.fill_(int(bool(g)))

    @property
    def supports_top_k_top_p(self) -> bool:
        """Whether add_request accepts top-k / top-p requests: the fused sampling head has no filter stage."""
        return not self.fused_head

    @property
    def ignore_eos(self) -> bool:
        return self._ignore_eos

    @ignore_eos.setter
    def ignore_eos(self, v: bool) -> None:
        self._ignore_eos = bool(v)
        self.ignore_eos_rows.fill_(int(bool(v)))

    # ------------------------------------------------------------------------------------------
    def _plan_gemms(self) -> None:
        cfg, B = self.cfg, self.B
        shapes = {"qkv": (cfg.qkv_size, cfg.hidden_size), "o": (cfg.hidden_size, cfg.q_size),
                  "gate_up": (2 * cfg.intermediate_size, cfg.hidden_size),
                  "down": (cfg.hidden_size, cfg.intermediate_size), "head": (cfg.head_rows, cfg.hidden_size)}
        self.split_k = {k: int(self.lib.prl_gemm_auto_split_k(B, n, kk)) for k, (n, kk) in shapes.items()}
        self.split_k["head"] = 1  # the sampler reads plain logits
        need = max(self.split_k[k] * B * shapes[k][0] for k in ("qkv", "o", "gate_up", "down"))
        self.partials = torch.zeros(need, dtype=torch.float32, device=self.dev)

    def _make_state(self) -> _lib.EngineState:
        s = _lib.EngineState()
        s.B = self.B
        s.sampled, s.sampled_logprobs = self.sampled.data_ptr(), self.sampled_lp.data_ptr()
        s.tokens, s.positions, s.seq_lens = self.tokens.data_ptr(), self.positions.data_ptr(), self.seq_lens.data_ptr()
        s.active = self.active.data_ptr()
        s.prompt_buf, s.prompt_stride, s.prompt_len = self.prompt_buf.data_ptr(), self.prompt_stride, self.prompt_len.data_ptr()
        s.out_ids, s.out_logprobs, s.out_stride = self.out_ids.data_ptr(), self.out_logprobs.data_ptr(), self.max_new
        s.gen_count, s.max_new, s.finished = self.gen_count.data_ptr(), self.max_new_t.data_ptr(), self.finished.data_ptr()
        s.eos_id, s.ignore_eos = self.eos_id, 0
        s.ignore_eos_rows = self.ignore_eos_rows.data_ptr()
        return s

    # ------------------------------------------------------------------------------------------
    def _gemm(self, w_name: str, x: torch.Tensor, n: int, k: int, split: int, out: torch.Tensor, lo: str | None = None,
              m: int | None = None):
        _lib.check(self.lib.prl_gemm_bf16_splitk(self.arena.ptr(w_name), self.arena.ptr(lo) if lo else None,
                                                 x.data_ptr(), self.B if m is None else m, n, k, split,
                                                 out.data_ptr(), self._st))

    def _step_kernels(self) -> None:
        """Enqueue one token step for all B slots on the current stream (graph-capturable)."""
        cfg, lib, B, a = self.cfg, self.lib, self.B, self.arena
        self._st = _lib.stream_ptr()
        st = self._st
        H, I = cfg.hidden_size, cfg.intermediate_size
        part = self.partials
        skip = self._skip
        pf = self.l2_prefetch_bytes  # cross-kernel L2 prefetch budget per site (0 disables)
        fuse_swiglu = (self.fuse_swiglu and not skip and not pf and self.split_k["gate_up"] == 1 and I % 64 == 0 and B <= 128)

        def wbytes(name):  # whole weight tensor, capped by the budget
            shape = a.layout.shapes[name]
            return min(pf, shape[0] * shape[1] * 2) if pf else 0
        _lib.check(lib.prl_embed_rmsnorm(self.tokens.data_ptr(), a.ptr("embed_tokens.weight"),
                                         a.ptr("layers.0.input_layernorm.weight"), cfg.rms_eps, B, H, cfg.vocab_size,
                                         self.h.data_ptr(), self.x.data_ptr(), st))
        sm_scale = 1.0 / math.sqrt(cfg.head_dim)
        for l in range(cfg.num_layers):
            p = f"layers.{l}."
            if "gemm" not in skip:
                self._gemm(p + "qkv_proj.weight", self.x, cfg.qkv_size, H, self.split_k["qkv"], part)
            if "small" not in skip:
                # while attention streams the KV cache, L2 fetches o_proj's weights
                _lib.check(lib.prl_qkv_rope_cache(part.data_ptr(), self.split_k["qkv"], B,
                                                  a.ptr(p + "qkv_proj.bias") if cfg.qkv_bias else None, cfg.num_q_heads,
                                                  cfg.num_kv_heads, cfg.head_dim, self.positions.data_ptr(),
                                                  self.block_table.data_ptr(), self.max_blocks, None,
                                                  self.inv_freq.data_ptr(), self.q.data_ptr(), self.kv_cache.data_ptr(),
                                                  self.n_pages, l, PAGE_SIZE,
                                                  a.ptr(p + "o_proj.weight") if pf else None, wbytes(p + "o_proj.weight"), st))
            if "attn" not in skip:
                _lib.check(lib.prl_paged_attn_decode(self.q.data_ptr(), self.kv_cache.data_ptr(), self.n_pages,
                                                     cfg.num_layers, l, self.block_table.data_ptr(), self.max_blocks,
                                                     self.seq_lens.data_ptr(), B, cfg.num_q_heads, cfg.num_kv_heads,
                                                     cfg.head_dim, PAGE_SIZE, self.attn_splits, sm_scale,
                                                     self.attn_out.data_ptr(), self.attn_ws.data_ptr(),
                                                     self.attn_ws.numel(), st))
            if "gemm" not in skip:
                self._gemm(p + "o_proj.weight", self.attn_out, H, cfg.q_size, self.split_k["o"], part)
            if "small" not in skip:
                # while gate_up streams, L2 fetches the head of down_proj
                _lib.check(lib.prl_residual_rmsnorm(part.data_ptr(), self.split_k["o"], B, H,
                                                    a.ptr(p + "post_attention_layernorm.weight"), cfg.rms_eps,
                                                    self.h.data_ptr(), self.x.data_ptr(),
                                                    a.ptr(p + "down_proj.weight") if pf else None,
                                                    wbytes(p + "down_proj.weight"), st))
            nxt_qkv = f"layers.{l + 1}.qkv_proj.weight" if l + 1 < cfg.num_layers else None
            if fuse_swiglu:
                # SiLU(gate) * up in the gate_up GEMM's epilogue (no split-K here: 2 I / 128 tiles fill the SMs): one launch
                # less per layer and no [B, 2 I] fp32 tile between the two; same bits as the pair below
                _lib.check(lib.prl_gemm_swiglu_decode(a.ptr(p + "gate_up_proj.weight"), self.x.data_ptr(), B, I, H,
                                                      self.act.data_ptr(), st))
            else:
                if "gemm" not in skip:
                    self._gemm(p + "gate_up_proj.weight", self.x, 2 * I, H, self.split_k["gate_up"], part)
                if "small" not in skip:
                    # while down streams, L2 fetches the next layer's qkv_proj
                    _lib.check(lib.prl_silu_mul(part.data_ptr(), self.split_k["gate_up"], B, I, self.act.data_ptr(),
                                                a.ptr(nxt_qkv) if (pf and nxt_qkv) else None,
                                                wbytes(nxt_qkv) if nxt_qkv else 0, st))
            if "gemm" not in skip:
                self._gemm(p + "down_proj.weight", self.act, H, I, self.split_k["down"], part)
            nxt = f"layers.{l + 1}.input_layernorm.weight" if l + 1 < cfg.num_layers else "norm.weight"
            if "small" not in skip:
                _lib.check(lib.prl_residual_rmsnorm(part.data_ptr(), self.split_k["down"], B, H, a.ptr(nxt), cfg.rms_eps,
                                                    self.h.data_ptr(), self.x.data_ptr(), None, 0, st))
        if not self.fused_head:
            self._gemm("lm_head.weight", self.x, cfg.head_rows, H, 1, self.logits,
                       lo="lm_head.weight_lo" if cfg.fp32_head else None)

    def _sample_and_advance(self) -> None:
        lib, st = self.lib, _lib.stream_ptr()
        if self.fused_head:
            cfg, a = self.cfg, self.arena
            _lib.check(lib.prl_head_logprob(a.ptr("lm_head.weight"), a.ptr("lm_head.weight_lo") if cfg.fp32_head else None,
                                            self.x.data_ptr(), self.B, cfg.vocab_size, cfg.hidden_size,
                                            float(self.temperature), None, int(self.greedy), self.seed, self.step_count,
                                            None, None, None, self.sampled.data_ptr(), self.sampled_lp.data_ptr(),
                                            self.head_ws.data_ptr(), self.head_ws.numel(), st))
            _lib.check(lib.prl_advance_state(C.byref(self._state), st))
            return
        _lib.check(lib.prl_sample_logprob_rows(self.logits.data_ptr(), self.B, self.cfg.head_rows,
                                               self.inv_temp_rows.data_ptr(), self.greedy_rows.data_ptr(), self.seed,
                                               self.step_count, self.sampled.data_ptr(), self.sampled_lp.data_ptr(),
                                               self.sample_ws.data_ptr(), self.sample_ws.numel(), st))
        if self._n_filtered > 0:
            # rewrites id / logprob of the filtered slots only; every other slot keeps the sample drawn above
            _lib.check(lib.prl_sample_filter_rows(self.logits.data_ptr(), self.B, self.cfg.head_rows,
                                                  self.inv_temp_rows.data_ptr(), self.greedy_rows.data_ptr(),
                                                  self.top_k_rows.data_ptr(), self.top_p_rows.data_ptr(), self.seed,
                                                  self.step_count, self.sampled.data_ptr(), self.sampled_lp.data_ptr(),
                                                  None, None, 0, st))
        _lib.check(lib.prl_advance_state(C.byref(self._state), st))

    def step(self) -> None:
        """One token for every active slot.  The model part is replayed from a CUDA graph; sampling and
        state advance are launched per step (they take the step counter as an RNG argument)."""
        if self._prefill_queue:
            if self.profile_timing:
                import time
                torch.cuda.current_stream().synchronize()
                t0 = time.perf_counter()
                self.run_prefill()
                torch.cuda.current_stream().synchronize()
                self.stats["prefill_s"] = self.stats.get("prefill_s", 0.0) + time.perf_counter() - t0
            else:
                self.run_prefill()
        if self.use_graph:
            key = self.arena.data.data_ptr()
            g = self._graphs.get(key)
            if g is None:
                self._step_kernels()  # warm-up outside capture (sets kernel attributes)
                torch.cuda.current_stream().synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._step_kernels()
                self._graphs[key] = g
            g.replay()
        else:
            self._step_kernels()
        self._sample_and_advance()
        self.step_count += 1

    def set_arena(self, arena: ParamArena) -> None:
        """Switch the parameter buffer between two token steps (weight update flip).  Graphs are cached per
        buffer, so after the first use of each of the two buffers a flip costs one dictionary lookup.
        Prompt pages cached for prefix sharing hold KV computed under the OLD weights: they are dropped from the cache
        (in-flight sequences keep their own references and finish on the KV they have, as in the reference, where
        running requests survive `receive_weight_update`, vllm1.py:158-182), so a request stamped with the new
        model_version never attends to stale prompt KV."""
        if arena is not self.arena:
            self.invalidate_prefix_cache()
        self.arena = arena

    def invalidate_prefix_cache(self) -> None:
        for h, pg in list(self._page_of_hash.items()):
            self._drop_cached_page(h, pg)

    def _drop_cached_page(self, h: int, pg: int) -> None:
        self._page_of_hash.pop(h, None)
        self._hash_of_page.pop(pg, None)
        self._tokens_of_page.pop(pg, None)
        self._page_pending.pop(pg, None)
        self.page_ref[pg] -= 1                     # the cache's own reference
        if self.page_ref[pg] == 0:
            self.free_pages.append(pg)

    def _check_token_ids(self, ids) -> None:
        lo, hi = min(ids), max(ids)
        if lo < 0 or hi >= self.cfg.vocab_size:
            raise ValueError(f"token id out of range [0, {self.cfg.vocab_size}): min {lo}, max {hi}")

    # ---- chunked prefill ------------------------------------------------------------------------
    def _prefill_buffers(self):
        if self._pf is None:
            cfg, C, d = self.cfg, self.prefill_chunk, self.dev
            H, I = cfg.hidden_size, cfg.intermediate_size
            widest = max(cfg.qkv_size, 2 * I, H)
            i32 = dict(dtype=torch.int32, device=d)
            self._pf = dict(
                tokens=torch.zeros(C, **i32), pos=torch.zeros(C, **i32), slot=torch.zeros(C, **i32),
                seq=torch.zeros(4, C, **i32),  # q_start, q_len, pos0, slot per packed sequence
                h=torch.zeros(C, H, dtype=torch.float32, device=d), x=torch.zeros(C, H, dtype=torch.bfloat16, device=d),
                q=torch.zeros(C, cfg.q_size, dtype=torch.bfloat16, device=d),
                attn=torch.zeros(C, cfg.q_size, dtype=torch.bfloat16, device=d),
                act=torch.zeros(C, I, dtype=torch.bfloat16, device=d),
                part=torch.zeros(C * widest, dtype=torch.float32, device=d))
        return self._pf

    def _prefill_rows(self, segs: list[tuple[Request, int, int]], score_temperature: float | None = None):
        """One packed chunk: segs = [(request, first prompt index, n tokens)], total rows <= prefill_chunk.
        With score_temperature, the fused head also returns log p(prompt[i+1] | prompt[:i+1]) for every row."""
        cfg, lib, a, pf = self.cfg, self.lib, self.arena, self._prefill_buffers()
        n = sum(k for _, _, k in segs)
        toks, pos, slot, meta = [], [], [], [[], [], [], []]
        at = 0
        for req, s0, k in segs:
            toks += req.prompt_ids[s0:s0 + k]
            pos += range(s0, s0 + k)
            slot += [req.slot] * k
            meta[0].append(at); meta[1].append(k); meta[2].append(s0); meta[3].append(req.slot)
            at += k
        pf["tokens"][:n].copy_(torch.tensor(toks, dtype=torch.int32), non_blocking=True)
        pf["pos"][:n].copy_(torch.tensor(pos, dtype=torch.int32), non_blocking=True)
        pf["slot"][:n].copy_(torch.tensor(slot, dtype=torch.int32), non_blocking=True)
        ns = len(segs)
        pf["seq"][:, :ns].copy_(torch.tensor(meta, dtype=torch.int32), non_blocking=True)
        self._st = _lib.stream_ptr()
        st, H, I = self._st, cfg.hidden_size, cfg.intermediate_size
        part, h, x = pf["part"], pf["h"], pf["x"]
        sm_scale = 1.0 / math.sqrt(cfg.head_dim)
        _lib.check(lib.prl_embed_rmsnorm(pf["tokens"].data_ptr(), a.ptr("embed_tokens.weight"),
                                         a.ptr("layers.0.input_layernorm.weight"), cfg.rms_eps, n, H, cfg.vocab_size,
                                         h.data_ptr(), x.data_ptr(), st))
        max_q = max(k for _, _, k in segs)
        big = n > 128   # compute-bound chunk: persistent CTA-pair GEMM; o/down accumulate straight into the fp32 residual

        def gemm(w_name, src, N, K, dst, accumulate=False):
            if big:
                _lib.check(lib.prl_gemm_tn(src.data_ptr(), K, a.ptr(w_name), K, n, N, K, dst.data_ptr(), N, 1,
                                           int(accumulate), None, None, 0, 1.0, st))
            else:
                self._gemm(w_name, src, N, K, 1, dst, m=n)

        def add_and_norm(gamma_name):
            # big: the GEMM epilogue already added its tile to h -> only the norm is left (zero partial slices)
            _lib.check(lib.prl_residual_rmsnorm(part.data_ptr(), 0 if big else 1, n, H, a.ptr(gamma_name), cfg.rms_eps,
                                                h.data_ptr(), x.data_ptr(), None, 0, st))
        for l in range(cfg.num_layers):
            p = f"layers.{l}."
            gemm(p + "qkv_proj.weight", x, cfg.qkv_size, H, part)
            _lib.check(lib.prl_qkv_rope_cache(part.data_ptr(), 1, n, a.ptr(p + "qkv_proj.bias") if cfg.qkv_bias else None,
                                              cfg.num_q_heads, cfg.num_kv_heads, cfg.head_dim, pf["pos"].data_ptr(),
                                              self.block_table.data_ptr(), self.max_blocks, pf["slot"].data_ptr(),
                                              self.inv_freq.data_ptr(), pf["q"].data_ptr(), self.kv_cache.data_ptr(),
                                              self.n_pages, l, PAGE_SIZE, None, 0, st))
            seq = pf["seq"]
            if self.prefill_attn_tc:   # tcgen05 path (csrc/attn_tc.cu)
                _lib.check(lib.prl_paged_attn_prefill_tc(pf["q"].data_ptr(), n, self.kv_cache.data_ptr(), self.n_pages,
                                                         cfg.num_layers, l, self.block_table.data_ptr(), self.max_blocks,
                                                         seq[0].data_ptr(), seq[1].data_ptr(), seq[2].data_ptr(),
                                                         seq[3].data_ptr(), ns, max_q, cfg.num_q_heads,
                                                         cfg.num_kv_heads, cfg.head_dim, PAGE_SIZE, sm_scale,
                                                         pf["attn"].data_ptr(), st))
            else:                      # mma.sync path (csrc/paged_attn.cu)
                _lib.check(lib.prl_paged_attn_prefill(pf["q"].data_ptr(), self.kv_cache.data_ptr(), self.n_pages,
                                                      cfg.num_layers, l, self.block_table.data_ptr(), self.max_blocks,
                                                      seq[0].data_ptr(), seq[1].data_ptr(), seq[2].data_ptr(),
                                                      seq[3].data_ptr(), ns, max_q, cfg.num_q_heads, cfg.num_kv_heads,
                                                      cfg.head_dim, PAGE_SIZE, sm_scale, pf["attn"].data_ptr(), st))
            gemm(p + "o_proj.weight", pf["attn"], H, cfg.q_size, h if big else part, accumulate=big)
            add_and_norm(p + "post_attention_layernorm.weight")
            if big and I % 128 == 0:
                # SiLU(gate) * up in the gate_up GEMM's epilogue, taken of the fp32 accumulators: the bits of the GEMM +
                # prl_silu_mul pair without the [n, 2 I] fp32 round trip through HBM (0.3 GB per layer and 1024-token chunk)
                _lib.check(lib.prl_gemm_swiglu_f32(x.data_ptr(), H, a.ptr(p + "gate_up_proj.weight"), H, n, I, H,
                                                   pf["act"].data_ptr(), I, st))
            else:
                gemm(p + "gate_up_proj.weight", x, 2 * I, H, part)
                _lib.check(lib.prl_silu_mul(part.data_ptr(), 1, n, I, pf["act"].data_ptr(), None, 0, st))
            gemm(p + "down_proj.weight", pf["act"], H, I, h if big else part, accumulate=big)
            add_and_norm(f"layers.{l + 1}.input_layernorm.weight" if l + 1 < cfg.num_layers else "norm.weight")
        self.stats["prefill_tokens"] += n
        if score_temperature is None:
            return None
        # teacher-forced scoring: targets = the next prompt token of every row; logits never reach HBM
        tg = []
        for req, s0, k in segs:
            tg += req.prompt_ids[s0 + 1:s0 + k + 1]
        if "targets" not in pf:
            pf["targets"] = torch.zeros(self.prefill_chunk, dtype=torch.int64, device=self.dev)
            pf["lp"] = torch.zeros(self.prefill_chunk, dtype=torch.float32, device=self.dev)
            pf["head_ws"] = torch.zeros(int(lib.prl_head_workspace_bytes(self.prefill_chunk, cfg.vocab_size)),
                                        dtype=torch.uint8, device=self.dev)
        pf["targets"][:n].copy_(torch.tensor(tg, dtype=torch.int64), non_blocking=True)
        _lib.check(lib.prl_head_logprob(a.ptr("lm_head.weight"), a.ptr("lm_head.weight_lo") if cfg.fp32_head else None,
                                        x.data_ptr(), n, cfg.vocab_size, H, float(score_temperature),
                                        pf["targets"].data_ptr(), 1, 0, 0, pf["lp"].data_ptr(), None, None, None, None,
                                        pf["head_ws"].data_ptr(), pf["head_ws"].numel(), st))
        return pf["lp"][:n].cpu().tolist()

    def score(self, sequences: list[list[int]], temperature: float = 1.0) -> list[list[float]]:
        """Teacher-forced log-probabilities log p(seq[i+1] | seq[:i+1]) — the reference-logprob path the
        preprocessor uses when kl_coef > 0 (`/v1/completions` with echo, pipelinerl/llm.py:606-648,
        preprocess.py:86-104) — through the chunked-prefill kernels and the fused head."""
        out: list[list[float]] = []
        for seq in sequences:
            n = len(seq)
            if n < 2:
                out.append([])
                continue
            if n > self.max_seq_len or not self.free_slots:
                raise RuntimeError("engine cannot score this sequence now (too long or no free slot)")
            req = Request(-1, list(seq), SamplingParams(max_tokens=0))
            req.slot = self.free_slots.pop()
            req.pages = self._alloc_pages((n + PAGE_SIZE - 1) // PAGE_SIZE)
            row = torch.zeros(self.max_blocks, dtype=torch.int32)
            row[:len(req.pages)] = torch.tensor(req.pages, dtype=torch.int32)
            self.block_table[req.slot].copy_(row, non_blocking=True)
            lps: list[float] = []
            at = 0
            while at < n - 1:
                k = min(self.prefill_chunk, n - 1 - at)
                lps += self._prefill_rows([(req, at, k)], score_temperature=temperature)
                at += k
            self.block_table[req.slot].zero_()
            self._release_pages(req.pages)
            self.free_slots.append(req.slot)
            out.append(lps)
        return out

    def run_prefill(self) -> int:
        """Prefill the not-yet-cached prompt tokens [start, P-1) of every queued request in packed chunks of
        <= prefill_chunk rows (the last prompt token goes through the decode step, which yields the first
        sample).  A request that shares prefix pages another queued request is still filling waits for them."""
        done = 0
        work = list(self._prefill_queue)
        self._prefill_queue = []
        C = self.prefill_chunk
        while work:
            segs, room = [], C
            progress_at_launch = {id(r): r.prefilled for r in work}
            for r in work:
                if room == 0:
                    break
                if any(progress_at_launch.get(id(o), o.prefilled) < need for o, need in r.waits_for):
                    continue
                k = min(room, len(r.prompt_ids) - 1 - r.prefilled)
                if k <= 0:
                    continue
                segs.append((r, r.prefilled, k))
                room -= k
            if not segs:
                raise RuntimeError("prefill scheduling deadlock (prefix dependency cycle)")
            self._prefill_rows(segs)
            for r, at, k in segs:
                r.prefilled = at + k
            done += sum(k for _, _, k in segs)
            work = [r for r in work if r.prefilled < len(r.prompt_ids) - 1]
        self._page_pending = {pg: (r, need) for pg, (r, need) in self._page_pending.items() if r.prefilled < need}
        return done

    # ---- pages and prefix sharing (page-granular, chained hashes: GRPO attempts AND later turns of a
    #      conversation reuse every full 64-token page of their common prefix) ------------------------------
    def _alloc_pages(self, n: int) -> list[int]:
        if len(self.free_pages) < n:
            self._evict_cached_pages(n - len(self.free_pages))
        if len(self.free_pages) < n:
            raise RuntimeError("engine out of KV pages")
        pages = [self.free_pages.pop() for _ in range(n)]
        for pg in pages:
            self.page_ref[pg] = 1
        return pages

    def _release_pages(self, pages: list[int]) -> None:
        for pg in pages:
            self.page_ref[pg] -= 1
            if self.page_ref[pg] == 0:
                self.free_pages.append(pg)

    def _evict_cached_pages(self, need: int) -> None:
        """Drop least-recently-used cached prefix pages that no live request references."""
        for h in list(self._page_of_hash):
            if need <= 0:
                break
            pg = self._page_of_hash[h]
            if self.page_ref[pg] == 1 and pg not in self._page_pending:
                self._drop_cached_page(h, pg)
                need -= 1

    def _evict_prefixes(self, need: int) -> None:  # kept name: tests / callers free the whole cache with a big `need`
        self._evict_cached_pages(need)

    @staticmethod
    def _page_hashes(prompt_ids: list[int], n_full: int) -> list[int]:
        out, h = [], 0
        for k in range(n_full):
            h = hash((h, tuple(prompt_ids[k * PAGE_SIZE:(k + 1) * PAGE_SIZE])))
            out.append(h)
        return out

    # ---- host-side admission / harvest --------------------------------------------------------
    def can_admit(self, prompt_len: int, max_tokens: int) -> bool:
        need = (prompt_len + max_tokens + PAGE_SIZE - 1) // PAGE_SIZE
        evictable = sum(1 for pg in self._hash_of_page if self.page_ref[pg] == 1 and pg not in self._page_pending)
        return bool(self.free_slots) and len(self.free_pages) + evictable >= need

    def add_request(self, prompt_ids: list[int], params: SamplingParams, model_version: int = 0) -> Request:
        n = len(prompt_ids)
        if n < 1:
            raise ValueError("empty prompt")
        if n + params.max_tokens > self.max_seq_len or params.max_tokens > self.max_new:
            raise ValueError(f"request of {n}+{params.max_tokens} tokens exceeds the engine limits")
        self._check_token_ids(prompt_ids)
        if not params.greedy and not params.temperature > 0:
            raise ValueError("temperature must be > 0 (use greedy=True for argmax)")
        params.check_filters()
        filtered = params.filtered(self.cfg.vocab_size)
        if filtered and not self.supports_top_k_top_p:
            raise ValueError("this engine has no top-k / top-p stage (the fused sampling head and the tensor-parallel "
                             "engine sample without one): serve top_k / top_p requests from a DecodeEngine built with "
                             "fused_head=False")
        if self.fused_head and (params.greedy != self._greedy or (not params.greedy and params.temperature != self._temperature)):
            raise ValueError("the fused sampling head takes engine-wide sampling parameters: build the engine with "
                             "fused_head=False to mix requests with different temperature / greedy settings")
        if not self.can_admit(n, params.max_tokens):
            raise RuntimeError("engine full")
        req = Request(self._next_id, list(prompt_ids), params, model_version=model_version)
        self._next_id += 1
        slot = self.free_slots.pop()
        n_pages = (n + params.max_tokens + PAGE_SIZE - 1) // PAGE_SIZE
        req.slot = slot
        start = 0  # index of the prompt token the decode loop processes first
        shared: list[int] = []
        if self.prefill_chunk > 0 and n > 1:
            start = n - 1
            n_full = (n - 1) // PAGE_SIZE
            hashes = self._page_hashes(prompt_ids, n_full) if self.prefix_sharing else []
            for k, h in enumerate(hashes):         # longest cached chain of full pages
                pg = self._page_of_hash.get(h)
                if pg is None:
                    break
                if self._tokens_of_page.get(pg) != tuple(prompt_ids[k * PAGE_SIZE:(k + 1) * PAGE_SIZE]):
                    break                          # hash collision: the cached page holds other tokens
                shared.append(pg)
                self._page_of_hash.move_to_end(h)
            for pg in shared:
                self.page_ref[pg] += 1
                if pg in self._page_pending:
                    owner, need = self._page_pending[pg]
                    req.waits_for.append((owner, need))
            own = self._alloc_pages(n_pages - len(shared))
            req.pages = shared + own
            req.prefilled = len(shared) * PAGE_SIZE
            for k in range(len(shared), len(hashes)):   # publish this request's own full prompt pages
                pg, h = req.pages[k], hashes[k]
                if h not in self._page_of_hash:
                    self._page_of_hash[h] = pg
                    self._hash_of_page[pg] = h
                    self._tokens_of_page[pg] = tuple(prompt_ids[k * PAGE_SIZE:(k + 1) * PAGE_SIZE])
                    self.page_ref[pg] += 1               # the cache's own reference
                    self._page_pending[pg] = (req, (k + 1) * PAGE_SIZE)
            if shared:
                self.stats["prefix_hits"] += 1
                self.stats["prefix_hit_tokens"] += len(shared) * PAGE_SIZE
            if req.prefilled < n - 1:
                self._prefill_queue.append(req)
        else:
            req.pages = self._alloc_pages(n_pages)
        row = torch.zeros(self.max_blocks, dtype=torch.int32)
        row[:n_pages] = torch.tensor(req.pages, dtype=torch.int32)
        self.block_table[slot].copy_(row, non_blocking=True)
        self.prompt_buf[slot, :n].copy_(torch.tensor(prompt_ids, dtype=torch.int32), non_blocking=True)
        self.prompt_len[slot] = n
        self.max_new_t[slot] = params.max_tokens
        self.inv_temp_rows[slot] = 1.0 if params.greedy else 1.0 / float(params.temperature)
        self.greedy_rows[slot] = int(bool(params.greedy))
        self.ignore_eos_rows[slot] = int(bool(params.ignore_eos) or self._ignore_eos)
        if filtered:
            req.filtered = True
            self.top_k_rows[slot] = params.top_k
            self.top_p_rows[slot] = params.top_p
            self._n_filtered += 1
        self.tokens[slot] = prompt_ids[start]
        self.positions[slot] = start
        self.seq_lens[slot] = start + 1
        self.gen_count[slot] = 0
        self.finished[slot] = 0
        self.active[slot] = 1
        self.slot_req[slot] = req
        return req

    def harvest(self) -> list[Request]:
        """Collect finished requests (one small D2H copy of the flags, then the finished rows)."""
        if not self.slot_req:
            return []
        fin = self.finished.cpu()
        done = []
        for slot, req in list(self.slot_req.items()):
            code = int(fin[slot])
            if code == 0:
                continue
            n = int(self.gen_count[slot].item())
            req.output_ids = self.out_ids[slot, :n].cpu().tolist()
            req.output_logprobs = self.out_logprobs[slot, :n].cpu().tolist()
            req.finish_reason = "stop" if code == 1 else "length"
            self.block_table[slot].zero_()
            self.finished[slot] = 0
            if req.filtered:
                self.top_k_rows[slot] = -1
                self.top_p_rows[slot] = 1.0
                self._n_filtered -= 1
            self._release_pages(req.pages)
            self.free_slots.append(slot)
            del self.slot_req[slot]
            done.append(req)
        return done

    def generate(self, prompts: list[list[int]], params: SamplingParams) -> list[Request]:
        """Convenience driver: run the given prompts to completion (used by tests and the bench)."""
        self.temperature, self.greedy, self.ignore_eos = params.temperature, params.greedy, params.ignore_eos
        pending = list(enumerate(prompts))
        results: dict[int, Request] = {}
        index_of: dict[int, int] = {}
        while pending or self.slot_req:
            while pending and self.can_admit(len(pending[0][1]), params.max_tokens):
                i, pr = pending.pop(0)
                r = self.add_request(pr, params)
                index_of[r.req_id] = i
            for _ in range(8):
                self.step()
            for r in self.harvest():
                results[index_of[r.req_id]] = r
        return [results[i] for i in range(len(prompts))]
