"""ctypes binding of libprl.so (include/prl.h).

The product path has no CPU fallback: if the library is missing this module
raises on first use.  Nothing under oracle/ is imported here.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "_lib" / "libprl.so"
_lib = None


class PrlError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libprl error {code}: {msg}")
        self.code = code


class NonFiniteError(AssertionError):
    """Mirrors the reference's `assert torch.isfinite(...)` (rl/__init__.py:213,263,291,386)."""


# ---- structs (field order = include/prl.h) -------------------------------------
class PgConfig(C.Structure):
    _fields_ = [
        ("policy_loss", C.c_int32), ("use_advantages", C.c_int32), ("relu_log_p_weights", C.c_int32),
        ("group_normalization", C.c_int32), ("overlong_filtering", C.c_int32), ("use_entropy_loss", C.c_int32),
        ("epsilon_low", C.c_float), ("epsilon_high", C.c_float), ("clamp_log_ratio_ref_new_value", C.c_float),
        ("kl_coef", C.c_float), ("entropy_bonus_coef", C.c_float), ("batch_size", C.c_float),
    ]


class PgBatch(C.Structure):
    _fields_ = [
        ("T", C.c_int64),
        ("new_logprobs", C.c_void_p), ("entropy", C.c_void_p), ("labels", C.c_void_p),
        ("rewards", C.c_void_p), ("advantages", C.c_void_p), ("ref_logprobs", C.c_void_p),
        ("old_logprobs", C.c_void_p), ("group_tokens", C.c_void_p), ("num_labels", C.c_void_p),
        ("overflow", C.c_void_p), ("segment_ids", C.c_void_p), ("position_ids", C.c_void_p),
        ("n_segments", C.c_int32), ("num_sequences", C.c_int32), ("sentinel", C.c_int32),
    ]


class AdamwArgs(C.Structure):
    _fields_ = [
        ("n", C.c_int64),
        ("master", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
        ("grad", C.c_void_p), ("grad_is_bf16", C.c_int32),
        ("param_bf16", C.c_void_p), ("param_bf16_lo", C.c_void_p),
        ("tensor_offsets", C.c_void_p), ("tensor_no_decay", C.c_void_p), ("n_tensors", C.c_int32),
        ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
        ("weight_decay", C.c_double), ("step", C.c_int32), ("max_grad_norm", C.c_float),
        ("grad_scale", C.c_float),
    ]


class AdamwShardArgs(C.Structure):
    _fields_ = [
        ("n", C.c_int64), ("shard_begin", C.c_int64), ("shard_end", C.c_int64),
        ("master", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
        ("grads", C.c_void_p * 8), ("shadows", C.c_void_p * 8), ("norm_tables", C.c_void_p * 8),
        ("n_peers", C.c_int32), ("rank", C.c_int32), ("grad_is_bf16", C.c_int32),
        ("gsum_scratch", C.c_void_p), ("tensor_offsets", C.c_void_p), ("tensor_no_decay", C.c_void_p),
        ("n_tensors", C.c_int32),
        ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double),
        ("step", C.c_int32), ("max_grad_norm", C.c_float), ("grad_scale", C.c_float),
    ]


class EngineState(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("sampled", C.c_void_p), ("sampled_logprobs", C.c_void_p), ("tokens", C.c_void_p),
        ("positions", C.c_void_p), ("seq_lens", C.c_void_p), ("active", C.c_void_p), ("prompt_buf", C.c_void_p),
        ("prompt_stride", C.c_int32), ("prompt_len", C.c_void_p), ("out_ids", C.c_void_p),
        ("out_logprobs", C.c_void_p), ("out_stride", C.c_int32), ("gen_count", C.c_void_p), ("max_new", C.c_void_p),
        ("finished", C.c_void_p), ("eos_id", C.c_int32), ("ignore_eos", C.c_int32), ("ignore_eos_rows", C.c_void_p),
    ]


class MbRecord(C.Structure):
    _fields_ = [("n_chunk", C.c_int32), ("n_pack", C.c_int32), ("padding", C.c_int32), ("total_tok", C.c_int32),
                ("total_lp", C.c_int32), ("n_stat_slots", C.c_int32), ("n_rollout_slots", C.c_int32), ("n_groups", C.c_int32),
                ("reward", C.c_void_p), ("stat_slot", C.c_void_p), ("rollout_slot", C.c_void_p), ("group_slot", C.c_void_p),
                ("n_tok_all", C.c_void_p), ("pack_idx", C.c_void_p), ("pack_flags", C.c_void_p), ("tok_off", C.c_void_p),
                ("lp_off", C.c_void_p), ("input_ids", C.c_void_p), ("labels", C.c_void_p), ("logprobs", C.c_void_p),
                ("ref_logprobs", C.c_void_p)]


class MbColumns(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("input_ids", "labels", "attention_mask", "position_ids", "segment_ids", "rewards",
                                          "advantages", "ref_logprobs", "old_logprobs", "group_tokens", "num_labels",
                                          "overflow", "seq_boundaries")]


PRL_NUM_STATS = 32
LOSS_IDS = {"ppo": 0, "reinforce": 1, "gspo": 2}
STAT_NAMES = [
    "loss", "max_loss", "min_loss", "reward", "max_reward", "min_reward", "entropy", "old_logprobs",
    "new_logprobs", "ref_logprobs", "advantage", "max_advantage", "min_advantage", "kl", "kl_new_old",
    "mean_abs_log_ratio_new_old", "max_kl", "min_kl", "ratio_new_old", "ratio_new_old_sum",
    "ratio_new_old_squared_sum", "ratio_ref_new", "ratio_ref_old", "clamp_log_ratio_ref_new_indicator",
    "clamp_log_ratio_new_old_indicator", "token_weight", "max_token_weight", "min_token_weight", "kl_coef",
    "entropy_bonus_coef", "num_output_tokens_sum", "input_size",
]
assert len(STAT_NAMES) == PRL_NUM_STATS

# symbol -> (restype, argtypes); every symbol include/prl.h declares must be listed here
_SIGNATURES = {
    "prl_last_error": (C.c_char_p, []),
    "prl_version": (C.c_int, []),
    "prl_launch_count": (C.c_uint64, []),
    "prl_set_pdl": (C.c_int, [C.c_int32]),
    "prl_attn_set_fused_combine": (C.c_int, [C.c_int32]),
    "prl_pg_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "prl_pg_loss_fwd_bwd": (C.c_int, [C.POINTER(PgBatch), C.POINTER(PgConfig), C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_pg_gspo_segment_sums": (C.c_int, [C.POINTER(PgBatch), C.POINTER(PgConfig), C.c_void_p, C.c_void_p]),
    "prl_pg_loss_fwd_bwd_seg": (C.c_int, [C.POINTER(PgBatch), C.POINTER(PgConfig), C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_logprob_tail_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_logprob_tail_bwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p]),
    "prl_gemm_auto_split_k": (C.c_int, [C.c_int64, C.c_int64, C.c_int64]),
    "prl_gemm_set_smem_budget_kb": (C.c_int, [C.c_int32]),
    "prl_gemm_set_tiled_weights": (C.c_int, [C.c_int32]),
    "prl_gemm_set_cta_pair": (C.c_int, [C.c_int32]),
    "prl_gemm_tn": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                              C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                              C.c_float, C.c_void_p]),
    "prl_rowops_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "prl_rmsnorm_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_float, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "prl_rmsnorm_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_colsum_bf16": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t,
                                  C.c_void_p]),
    "prl_rope_inplace": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_float, C.c_void_p]),
    "prl_silu_mul_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "prl_silu_mul_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "prl_embed_gather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "prl_embed_scatter_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "prl_gemm_ex": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64,
                              C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                              C.c_float, C.c_void_p]),
    "prl_transpose_bf16": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "prl_gemm_bf16_splitk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                       C.c_void_p, C.c_void_p]),
    "prl_head_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "prl_head_logprob": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_float,
                                   C.c_void_p, C.c_int32, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_embed_rmsnorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_residual_rmsnorm": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_qkv_rope_cache": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_paged_attn_prefill_tc": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                            C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                            C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                            C.c_void_p, C.c_void_p]),
    "prl_attn_varlen_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_attn_set_fwd_generation": (C.c_int, [C.c_int32]),
    "prl_attn_set_bwd_generation": (C.c_int, [C.c_int32]),
    "prl_attn_set_prefill_generation": (C.c_int, [C.c_int32]),
    "prl_debug_tmem_read_bench": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "prl_attn_debug_timing": (C.c_int, [C.c_void_p]),
    "prl_attn_debug_bwd_timing": (C.c_int, [C.c_void_p]),
    "prl_attn_debug_bwd_timing_dkdv": (C.c_int, [C.c_void_p]),
    "prl_debug_mma_bench": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "prl_attn_varlen_bwd_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "prl_attn_varlen_fwd_kv": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_attn_varlen_bwd_kv": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_attn_varlen_bwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_paged_attn_prefill": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                         C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                         C.c_void_p, C.c_void_p]),
    "prl_silu_mul": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                               C.c_void_p]),
    "prl_paged_attn_splits": (C.c_int, [C.c_int32, C.c_int32, C.c_int32]),
    "prl_paged_attn_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "prl_paged_attn_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                        C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_void_p]),
    "prl_sample_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "prl_sample_logprob": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_uint64,
                                     C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_gemm_swiglu": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p,
                                  C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "prl_gemm_swiglu_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "prl_gemm_dgrad_swiglu": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                        C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "prl_gemm_swiglu_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                      C.c_void_p, C.c_int64, C.c_void_p]),
    "prl_bf16_residual": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "prl_preprocess_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "prl_preprocess_pack": (C.c_int, [C.POINTER(MbRecord), C.c_int32, C.c_int32, C.POINTER(MbColumns), C.c_void_p,
                                      C.c_size_t, C.c_void_p]),
    "prl_sample_logprob_rows": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64,
                                          C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_sample_filter_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "prl_sample_filter_rows": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_void_p]),
    "prl_advance_state": (C.c_int, [C.POINTER(EngineState), C.c_void_p]),
    "prl_gemm_bf16_splitk_peer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_tp_signal": (C.c_int, [C.c_void_p, C.c_void_p]),
    "prl_tp_wait": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "prl_tp_epoch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "prl_sample_partials": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_uint64, C.c_uint32,
                                      C.c_int32, C.c_void_p, C.c_void_p]),
    "prl_sample_finalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "prl_ipc_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "prl_ipc_free": (C.c_int, [C.c_void_p]),
    "prl_ipc_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "prl_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "prl_ipc_close": (C.c_int, [C.c_void_p]),
    "prl_enable_peer_access": (C.c_int, [C.c_int32]),
    "prl_weights_push": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_size_t, C.c_size_t, C.c_int32,
                                   C.c_void_p]),
    "prl_weights_signal": (C.c_int, [C.POINTER(C.c_void_p), C.c_int32, C.c_uint64, C.c_void_p]),
    "prl_logprob_rows_bwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_float,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.c_void_p]),
    "prl_head_dlogits": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "prl_adamw_sharded_reduce": (C.c_int, [C.POINTER(AdamwShardArgs), C.c_void_p, C.c_size_t, C.c_void_p]),
    "prl_adamw_sharded_update": (C.c_int, [C.POINTER(AdamwShardArgs), C.c_void_p, C.c_void_p]),
    "prl_adamw_workspace_bytes": (C.c_size_t, []),
    "prl_adamw_step": (C.c_int, [C.POINTER(AdamwArgs), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}


def lib_path() -> Path:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load libprl.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise RuntimeError(
                f"{_LIB_PATH} is missing: build it with `python -m pipelinerl_b200._build` "
                "(the CUDA extension is the product; there is no CPU fallback)")
        lib = C.CDLL(str(_LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def declared_symbols() -> list[str]:
    return sorted(_SIGNATURES)


def check(code: int) -> None:
    if code != 0:
        msg = load().prl_last_error().decode(errors="replace")
        raise PrlError(code, msg)


def launch_count() -> int:
    return int(load().prl_launch_count())


def stream_ptr(stream=None) -> int:
    """cudaStream_t of a torch stream (current stream by default) as an integer."""
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return int(s.cuda_stream)
