"""Tensor-parallel sampler engine (BASELINE config 4: Qwen2.5-32B, TP=2 inference).

One process per GPU, SPMD: every rank of a TP group runs the same admission / step sequence (a serving
deployment would broadcast the leader's scheduling decisions; tests and the bench drive the ranks in lockstep).
Sharding: column-parallel qkv / gate_up / lm_head, row-parallel o_proj / down_proj, local attention over this
rank's kv heads, replicated embeddings and norms (`ModelConfig.shard`).

No NCCL on the token path.  A row-parallel GEMM writes its fp32 split-K partial tiles into its own AND its peers'
reduction buffers from the GEMM epilogue (P2P stores over NVLink, `prl_gemm_bf16_splitk_peer`); a counter in peer
memory orders producer and consumer (`prl_tp_signal` / `prl_tp_wait`); the ordinary split reduction of
`prl_residual_rmsnorm` then sums tp x split slots in a fixed order, so all ranks hold bit-identical residual
streams.  The vocab-parallel head exchanges 16 sampler partials per row (512 B) instead of logits.
The reference delegates this to vLLM's tensor-parallel-size (world.py:56-59; NCCL / custom all-reduce twice
per layer).
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from .engine import PAGE_SIZE, DecodeEngine
from .model import ModelConfig, ParamArena
from .weights import ipc_alloc, ipc_export, ipc_open


class TPDecodeEngine(DecodeEngine):
    def __init__(self, full_cfg: ModelConfig, arena: ParamArena, tp_rank: int, tp_size: int, group=None, **kw):
        import torch.distributed as dist
        if tp_size < 2 or tp_size > 8:
            raise ValueError("TPDecodeEngine is for 2..8 ranks; use DecodeEngine for tp=1")
        self.full_cfg, self.tp_rank, self.tp, self.dist, self.group = full_cfg, tp_rank, tp_size, dist, group
        kw["prefill_chunk"] = 0          # prompts go through the decode path (TP chunked prefill: next step)
        kw["fused_head"] = False
        super().__init__(full_cfg.shard(tp_size), arena, **kw)
        cfg, B, H = self.cfg, self.B, self.cfg.hidden_size
        self.tp_split = {"o": self.split_k["o"], "down": self.split_k["down"]}
        s_max = max(self.tp_split.values())
        self._slot_elems = s_max * B * H                        # one rank's partials of one GEMM
        self._buf_elems = self.tp * self._slot_elems             # [tp][S][B][H]
        # IPC memory of this rank: two reduction buffers (o_proj / down_proj), sampler exchange, counters
        self._part_buf = ipc_alloc(2 * self._buf_elems * 4)
        self._samp_buf = ipc_alloc(self.tp * B * 16 * 32)
        self._flag_buf = ipc_alloc(64)                           # [0] = deliveries received from each peer (one counter per peer)
        self.tp_part = self._part_buf.tensor(torch.float32, self.dev)
        self.tp_samp = self._samp_buf.tensor(torch.uint8, self.dev)
        self.tp_flags = self._flag_buf.tensor(torch.int64, self.dev)
        self.tp_epoch = torch.zeros(1, dtype=torch.int64, device=self.dev)
        mine = (ipc_export(self._part_buf), ipc_export(self._samp_buf), ipc_export(self._flag_buf))
        gathered = [None] * self.tp
        dist.all_gather_object(gathered, mine, group=group)
        self._peer_bufs, self._peer_part, self._peer_samp, self._peer_flag = [], {}, {}, {}
        for r, (hp, hs, hf) in enumerate(gathered):
            if r == tp_rank:
                continue
            bp, bs, bf = ipc_open(hp, 2 * self._buf_elems * 4), ipc_open(hs, self.tp * B * 16 * 32), ipc_open(hf, 64)
            self._peer_bufs += [bp, bs, bf]
            self._peer_part[r], self._peer_samp[r], self._peer_flag[r] = bp.ptr, bs.ptr, bf.ptr
        if self.tp != 2:
            raise NotImplementedError("peer-store epilogue currently targets one peer (tp=2, BASELINE config 4)")
        self.peer = 1 - tp_rank
        self._eager_done: set[int] = set()
        self.signals_per_step = 2 * cfg.num_layers + 1
        dist.barrier(group=group)

    # slot of rank r in reduction buffer `which` (0 = o_proj, 1 = down_proj)
    def _slot(self, base_ptr: int, which: int, r: int) -> int:
        return base_ptr + (which * self._buf_elems + r * self._slot_elems) * 4

    def _row_parallel(self, w_name: str, x: torch.Tensor, n: int, k: int, which: int, split: int, sync_k: int,
                      gamma_ptr: int, prefetch=(None, 0)) -> None:
        """Row-parallel GEMM with the all-reduce fused into its epilogue, then residual + RMSNorm over tp x split slots."""
        lib, st, B = self.lib, self._st, self.B
        local = self._slot(self._part_buf.ptr, which, self.tp_rank)
        remote = self._slot(self._peer_part[self.peer], which, self.tp_rank)
        _lib.check(lib.prl_gemm_bf16_splitk_peer(self.arena.ptr(w_name), x.data_ptr(), B, n, k, split, local, remote, st))
        _lib.check(lib.prl_tp_signal(self._peer_flag[self.peer], st))
        _lib.check(lib.prl_tp_wait(self._flag_buf.ptr, self.tp_epoch.data_ptr(), self.signals_per_step, sync_k, st))
        # slots [rank 0 splits | rank 1 splits] are contiguous only when split == s_max; reduce each rank's block
        base = self._slot(self._part_buf.ptr, which, 0)
        if split * self.B * self.cfg.hidden_size == self._slot_elems:
            _lib.check(lib.prl_residual_rmsnorm(base, self.tp * split, B, self.cfg.hidden_size, gamma_ptr,
                                                self.cfg.rms_eps, self.h.data_ptr(), self.x.data_ptr(), None, 0, st))
        else:
            raise RuntimeError("reduction slots must be dense (split == s_max)")

    def _step_kernels(self) -> None:
        cfg, lib, B, a = self.cfg, self.lib, self.B, self.arena
        self._st = _lib.stream_ptr()
        st, H, I = self._st, cfg.hidden_size, cfg.intermediate_size
        part = self.partials
        _lib.check(lib.prl_embed_rmsnorm(self.tokens.data_ptr(), a.ptr("embed_tokens.weight"),
                                         a.ptr("layers.0.input_layernorm.weight"), cfg.rms_eps, B, H, cfg.vocab_size,
                                         self.h.data_ptr(), self.x.data_ptr(), st))
        sm_scale = 1.0 / math.sqrt(cfg.head_dim)
        s_dense = self._slot_elems // (B * H)
        for l in range(cfg.num_layers):
            p = f"layers.{l}."
            self._gemm(p + "qkv_proj.weight", self.x, cfg.qkv_size, H, self.split_k["qkv"], part)
            _lib.check(lib.prl_qkv_rope_cache(part.data_ptr(), self.split_k["qkv"], B,
                                              a.ptr(p + "qkv_proj.bias") if cfg.qkv_bias else None, cfg.num_q_heads,
                                              cfg.num_kv_heads, cfg.head_dim, self.positions.data_ptr(),
                                              self.block_table.data_ptr(), self.max_blocks, None, self.inv_freq.data_ptr(),
                                              self.q.data_ptr(), self.kv_cache.data_ptr(), self.n_pages, l, PAGE_SIZE,
                                              None, 0, st))
            _lib.check(lib.prl_paged_attn_decode(self.q.data_ptr(), self.kv_cache.data_ptr(), self.n_pages, cfg.num_layers,
                                                 l, self.block_table.data_ptr(), self.max_blocks, self.seq_lens.data_ptr(),
                                                 B, cfg.num_q_heads, cfg.num_kv_heads, cfg.head_dim, PAGE_SIZE,
                                                 self.attn_splits, sm_scale, self.attn_out.data_ptr(),
                                                 self.attn_ws.data_ptr(), self.attn_ws.numel(), st))
            self._row_parallel(p + "o_proj.weight", self.attn_out, H, cfg.q_size, 0, s_dense, 2 * l + 1,
                               a.ptr(p + "post_attention_layernorm.weight"))
            self._gemm(p + "gate_up_proj.weight", self.x, 2 * I, H, self.split_k["gate_up"], part)
            _lib.check(lib.prl_silu_mul(part.data_ptr(), self.split_k["gate_up"], B, I, self.act.data_ptr(), None, 0, st))
            nxt = f"layers.{l + 1}.input_layernorm.weight" if l + 1 < cfg.num_layers else "norm.weight"
            self._row_parallel(p + "down_proj.weight", self.act, H, I, 1, s_dense, 2 * l + 2, a.ptr(nxt))
        self._gemm("lm_head.weight", self.x, cfg.head_rows, H, 1, self.logits)

    def step(self) -> None:
        """Like DecodeEngine.step, but the base class's eager warm-up before graph capture would deliver every
        peer signal twice in that step; here the first step of a parameter buffer runs eagerly AS the step (it also
        sets the kernel attributes) and the graph is captured, without a dry run, on the next one."""
        if self.use_graph:
            key = self.arena.data.data_ptr()
            g = self._graphs.get(key)
            if g is None:
                if key not in self._eager_done:
                    self._eager_done.add(key)
                    self._step_kernels()
                    self._sample_and_advance()
                    self.step_count += 1
                    return
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._step_kernels()
                self._graphs[key] = g
            g.replay()
        else:
            self._step_kernels()
        self._sample_and_advance()
        self.step_count += 1

    def _plan_gemms(self) -> None:
        super()._plan_gemms()
        # both row-parallel GEMMs use the same split so that the reduction slots are dense; every split is also a
        # P2P copy of the partial tile, so take the smallest split that still gives one CTA per SM
        tiles = (self.cfg.hidden_size + 127) // 128
        kb_o = (self.cfg.q_size + 63) // 64
        kb_d = (self.cfg.intermediate_size + 63) // 64
        s = max(1, -(-148 // tiles))
        s = max(1, min(s, kb_o // 4, kb_d // 4))
        self.split_k["o"] = self.split_k["down"] = s

    @property
    def supports_top_k_top_p(self) -> bool:
        """The vocab-parallel head merges sampler partials across ranks; it has no top-k / top-p stage."""
        return False

    def _sample_and_advance(self) -> None:
        lib, st, B, cfg = self.lib, _lib.stream_ptr(), self.B, self.cfg
        group_bytes = B * 16 * 32
        mine = self._samp_buf.ptr + self.tp_rank * group_bytes
        _lib.check(lib.prl_sample_partials(self.logits.data_ptr(), B, cfg.head_rows, float(self.temperature),
                                           int(self.greedy), self.seed, self.step_count, self.tp_rank * cfg.head_rows,
                                           mine, st))
        dst = (C.c_void_p * 1)(self._peer_samp[self.peer])
        _lib.check(lib.prl_weights_push(self._samp_buf.ptr, dst, 1, self.tp_rank * group_bytes, group_bytes, 4, st))
        _lib.check(lib.prl_tp_signal(self._peer_flag[self.peer], st))
        _lib.check(lib.prl_tp_wait(self._flag_buf.ptr, self.tp_epoch.data_ptr(), self.signals_per_step,
                                   self.signals_per_step, st))
        _lib.check(lib.prl_sample_finalize(self._samp_buf.ptr, B, self.tp, self.sampled.data_ptr(),
                                           self.sampled_lp.data_ptr(), st))
        self._state.ignore_eos = int(self.ignore_eos)
        _lib.check(lib.prl_advance_state(C.byref(self._state), st))
        _lib.check(lib.prl_tp_epoch(self.tp_epoch.data_ptr(), st))

    def close(self) -> None:
        torch.cuda.synchronize()
        self.dist.barrier(group=self.group)
        for b in self._peer_bufs:
            b.release()
        for b in (self._part_buf, self._samp_buf, self._flag_buf):
            b.release()
