/*
 * prl.h — C ABI of libprl.so, the B200 (sm_100a) hot-path library behind the
 * PipelineRL plugin / stream API.
 *
 * Conventions (SURVEY.md §8b):
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every device buffer is owned by the caller; the library owns only opaque
 *     handles it hands out from *_create and frees in *_destroy;
 *   - no allocation inside hot calls; every call takes an explicit stream
 *     (a cudaStream_t passed as void*; NULL = legacy default stream);
 *   - functions return 0 on success, <0 on error; prl_last_error() gives the
 *     message for the calling thread. Nothing throws across the ABI;
 *   - the library is not internally threaded: one host thread per GPU drives it.
 *
 * Each entry point cites the reference interface it replaces
 * (paths relative to the ServiceNow/PipelineRL tree).
 */
#ifndef PRL_H_
#define PRL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRL_OK 0
#define PRL_ERR_INVALID (-1)   /* bad argument */
#define PRL_ERR_CUDA (-2)      /* CUDA runtime / driver error */
#define PRL_ERR_UNSUPPORTED (-3)
#define PRL_ERR_NONFINITE (-4) /* reproduces the reference's isfinite asserts */

typedef void* prl_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------- */
const char* prl_last_error(void);
int prl_version(void);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
uint64_t prl_launch_count(void);
/* Tuning switches (A/B measurements): programmatic dependent launch on the token-step kernels (default on,
 * env PRL_PDL=0 disables) and in-kernel merge of the attention context splits (default off). */
int prl_set_pdl(int32_t on);
int prl_attn_set_fused_combine(int32_t on);

/* ======================================================================= *
 * Hot path (2a): policy-gradient loss tail
 *   replaces pipelinerl/finetune/rl/__init__.py:237-439 (rl_step after the
 *   logprob tail) and rl/utils.py:71-92 (sum_sum) — one launch instead of
 *   ~25 per-segment Python loops and ~30 .item() syncs.
 * ======================================================================= */

enum { PRL_LOSS_PPO = 0, PRL_LOSS_REINFORCE = 1, PRL_LOSS_GSPO = 2 };

/* index of each statistic in the stats[] output (order of rl/__init__.py:398-439) */
enum {
  PRL_STAT_LOSS = 0, PRL_STAT_MAX_LOSS, PRL_STAT_MIN_LOSS,
  PRL_STAT_REWARD, PRL_STAT_MAX_REWARD, PRL_STAT_MIN_REWARD,
  PRL_STAT_ENTROPY, PRL_STAT_OLD_LOGPROBS, PRL_STAT_NEW_LOGPROBS, PRL_STAT_REF_LOGPROBS,
  PRL_STAT_ADVANTAGE, PRL_STAT_MAX_ADVANTAGE, PRL_STAT_MIN_ADVANTAGE,
  PRL_STAT_KL, PRL_STAT_KL_NEW_OLD, PRL_STAT_MEAN_ABS_LOG_RATIO_NEW_OLD,
  PRL_STAT_MAX_KL, PRL_STAT_MIN_KL,
  PRL_STAT_RATIO_NEW_OLD, PRL_STAT_RATIO_NEW_OLD_SUM, PRL_STAT_RATIO_NEW_OLD_SQUARED_SUM,
  PRL_STAT_RATIO_REF_NEW, PRL_STAT_RATIO_REF_OLD,
  PRL_STAT_CLAMP_LOG_RATIO_REF_NEW_INDICATOR, PRL_STAT_CLAMP_LOG_RATIO_NEW_OLD_INDICATOR,
  PRL_STAT_TOKEN_WEIGHT, PRL_STAT_MAX_TOKEN_WEIGHT, PRL_STAT_MIN_TOKEN_WEIGHT,
  PRL_STAT_KL_COEF, PRL_STAT_ENTROPY_BONUS_COEF,
  PRL_STAT_NUM_OUTPUT_TOKENS_SUM, PRL_STAT_INPUT_SIZE,
  PRL_NUM_STATS /* = 32 */
};

/* RLConfig fields the loss tail reads (rl/__init__.py:43-105), with the decayed
 * coefficients already evaluated by the caller (linear_decay_coef, :119-133). */
typedef struct {
  int32_t policy_loss;          /* PRL_LOSS_* */
  int32_t use_advantages;       /* bool */
  int32_t relu_log_p_weights;   /* bool */
  int32_t group_normalization;  /* bool */
  int32_t overlong_filtering;   /* bool */
  int32_t use_entropy_loss;     /* bool: entropy_bonus != 0 or final_entropy_bonus != 0 */
  float epsilon_low, epsilon_high;
  float clamp_log_ratio_ref_new_value;
  float kl_coef;                /* already decayed for current_step */
  float entropy_bonus_coef;     /* already decayed */
  float batch_size;             /* config.batch_size (token weight = 1/batch_size) */
} prl_pg_config;

/* One packed row [1, T] (PipelineBatchEncoding, finetune/types.py:46-75). All
 * pointers are device pointers. Token-aligned columns are UNSHIFTED, length T;
 * the kernel applies the reference's [:, 1:] shift itself. new_logprobs and
 * entropy are the outputs of the logprob tail, length T-1 (position t holds the
 * log-probability of token t+1). */
typedef struct {
  int64_t T;                   /* tokens in the packed row (input_ids.numel()) */
  const float* new_logprobs;   /* [T-1] */
  const float* entropy;        /* [T-1] or NULL (treated as 0) */
  const int64_t* labels;       /* [T]  mask = labels[t+1] != -100 */
  const float* rewards;        /* [T] */
  const float* advantages;     /* [T] */
  const float* ref_logprobs;   /* [T] */
  const float* old_logprobs;   /* [T] */
  const float* group_tokens;   /* [T] */
  const float* num_labels;     /* [T] */
  const float* overflow;       /* [T] */
  const int64_t* segment_ids;  /* [T] or NULL; required for PRL_LOSS_GSPO */
  const int64_t* position_ids; /* [T] or NULL. When given, num_sequences is counted on the device as
                                  1 + #{t >= 1 : position_ids[t] == 0} (rl/__init__.py:166-178) */
  int32_t n_segments;          /* GSPO: any upper bound on max(segment_ids[1:]) + 1 (empty segments
                                  contribute nothing, as in the reference); else ignored */
  int32_t num_sequences;       /* used when position_ids is NULL (unpacked batch: number of rows) */
  int32_t sentinel;            /* batch.sentinel */
} prl_pg_batch;

/* Scratch the caller allocates once: prl_pg_workspace_bytes(max n_segments) bytes. */
size_t prl_pg_workspace_bytes(int32_t max_segments);

/* Forward + backward of the loss tail in one pass.
 *   loss          [1]  device, = final_loss (policy_loss_total)
 *   dloss_dlogprob[T-1] device, d final_loss / d new_logprobs (may be NULL)
 *   dloss_dentropy[T-1] device or NULL, d final_loss / d entropy (only non-zero
 *                       when use_entropy_loss)
 *   stats         [PRL_NUM_STATS] device doubles, the reference's stats dict;
 *                 when no token is labelled only PRL_STAT_INPUT_SIZE is meaningful
 *                 (rl/__init__.py:388-392) and PRL_STAT_NUM_OUTPUT_TOKENS_SUM is 0.
 *   nonfinite     [1] device int32: bitmask, bit0 new_logprobs, bit1 log_ratio_ref_new,
 *                 bit2 approx_kl, bit3 loss (the reference's asserts :213,263,291,386)
 */
int prl_pg_loss_fwd_bwd(const prl_pg_batch* batch, const prl_pg_config* cfg,
                        float* loss, float* dloss_dlogprob, float* dloss_dentropy,
                        double* stats, int32_t* nonfinite,
                        void* workspace, size_t workspace_bytes, prl_stream_t stream);

/* GSPO under sequence parallelism (rl/utils.py:194-206: the per-segment sums are all-reduced over the group).
 * Step 1 writes this rank's sums over its slice, seg_sums[n_segments][4] doubles = (sum log-ratio new/old, sum advantage,
 * token count, sum token weight); the caller SUM-all-reduces the array over the group.  Step 2 is prl_pg_loss_fwd_bwd with
 * those totals given; seg_local_count[n_segments] (this rank's token counts, or NULL) scales every segment's loss term to
 * this rank's share so that the ranks' losses add up to the loss of the whole row. */
int prl_pg_gspo_segment_sums(const prl_pg_batch* batch, const prl_pg_config* cfg, double* seg_sums, prl_stream_t stream);
int prl_pg_loss_fwd_bwd_seg(const prl_pg_batch* batch, const prl_pg_config* cfg, float* loss, float* dloss_dlogprob,
                            float* dloss_dentropy, double* stats, int32_t* nonfinite, void* workspace,
                            size_t workspace_bytes, const double* seg_sums, const double* seg_local_count,
                            prl_stream_t stream);

/* ======================================================================= *
 * Hot path (2b, generic-model variant): logprob tail from materialised logits
 *   replaces pipelinerl/finetune/rl/__init__.py:207-233 (logits/T, gather,
 *   logsumexp, 38-chunk entropy) with one read of the logits; backward reads
 *   once, writes once.  logits [T, V] fp32 with row stride `row_stride`
 *   elements; outputs have T-1 entries (position t scores token t+1).
 * ======================================================================= */
int prl_logprob_tail_fwd(const float* logits, int64_t T, int64_t V, int64_t row_stride,
                         const int64_t* input_ids, float temperature,
                         float* new_logprobs /*[T-1]*/, float* entropy /*[T-1] or NULL*/,
                         float* lse /*[T-1] or NULL, saved for backward*/, prl_stream_t stream);
/* dlogits [T, V] (row T-1 is zero-filled).  g_entropy may be NULL. */
int prl_logprob_tail_bwd(const float* logits, int64_t T, int64_t V, int64_t row_stride,
                         const int64_t* input_ids, float temperature,
                         const float* lse, const float* entropy,
                         const float* g_logprobs, const float* g_entropy,
                         float* dlogits, int64_t dlogits_stride, prl_stream_t stream);

/* Same backward for an explicit list of rows with their targets (logits [n_rows, V] of a recomputed chunk). */
int prl_logprob_rows_bwd(const float* logits, int64_t n_rows, int64_t V, int64_t row_stride,
                         const int64_t* targets /*[n_rows]*/, float temperature, const float* lse,
                         const float* entropy, const float* g_logprobs, const float* g_entropy,
                         float* dlogits, int64_t dlogits_stride, prl_stream_t stream);
/* Backward of the fused head WITHOUT materialised logits: one GEMM (X W_hi^T + X W_lo^T in TMEM, as prl_head_logprob) whose
 * epilogue writes dz[M, ld_dz] bf16 = inv_T * (g_lp * (onehot(target) - p) - g_ent * p * (log p + H)), p = exp(z / T - lse):
 * the operand of the dX / dW GEMMs.  Replaces logits GEMM(s) -> prl_logprob_rows_bwd -> bf16 cast (autograd through
 * rl/__init__.py:207-233).  lse / entropy: the forward's outputs; g_logprobs / g_entropy may be NULL. */
int prl_head_dlogits(const void* W_bf16, const void* W_lo_bf16, const void* X_bf16, int64_t M, int64_t V, int64_t K,
                     float temperature, const int64_t* targets, const float* lse, const float* entropy,
                     const float* g_logprobs, const float* g_entropy, void* dz_bf16, int64_t ld_dz, prl_stream_t stream);

/* ======================================================================= *
 * Hot path (2c): fused AdamW over a flat parameter arena
 *   replaces torch.optim.AdamW as built by pipelinerl/finetune/optim.py:25-29
 *   + clip_grad_norm_ (finetune_loop.py:739) + the bf16 re-cast of the
 *   DeepSpeed bf16 optimizer (finetune_loop.py:727-736).
 * ======================================================================= */
typedef struct {
  int64_t n;                 /* elements in the arena */
  float* master;             /* [n] fp32 master weights (in/out) */
  float* exp_avg;            /* [n] (in/out) */
  float* exp_avg_sq;         /* [n] (in/out) */
  const void* grad;          /* [n] bf16 or fp32 gradient */
  int32_t grad_is_bf16;
  void* param_bf16;          /* [n] bf16 copy consumed by fwd/bwd and the weight push (out), or NULL */
  void* param_bf16_lo;       /* [n] bf16 residual master - bf16(master) (out) or NULL: fp32-equivalent head */
  /* weight-decay groups (optim.py:8-22): tensor t covers [tensor_offsets[t], tensor_offsets[t+1]) */
  const int64_t* tensor_offsets; /* device [n_tensors+1], ascending, [0]=0, [n_tensors]=n */
  const uint8_t* tensor_no_decay;/* device [n_tensors] 1 = weight_decay 0 (bias / LayerNorm.weight) */
  int32_t n_tensors;
  double lr, beta1, beta2, eps, weight_decay; /* doubles: torch derives 1-beta, lr*wd, bias corrections in double */
  int32_t step;              /* 1-based optimizer step (bias correction) */
  float max_grad_norm;       /* <=0: no clipping */
  float grad_scale;          /* gradients are multiplied by this before use (1/accum etc.); 1.0 default */
} prl_adamw_args;

size_t prl_adamw_workspace_bytes(void);
/* grad_norm_out: device float[1], the pre-clip global L2 norm (as clip_grad_norm_ returns). */
int prl_adamw_step(const prl_adamw_args* args, float* grad_norm_out,
                   void* workspace, size_t workspace_bytes, prl_stream_t stream);

/* lo = bf16(master - float(bf16(master))) for n elements, stored to n_dst (<= 8) destinations (own arena tail and, under
 * data parallelism, the peers' over NVLink).  With hi = bf16(master) (the ordinary bf16 parameter) the pair is the
 * fp32-equivalent lm_head the reference computes on both sides (vllm_quantization.py:266-278, checkpoints.py:44-105):
 * prl_head_logprob / prl_gemm_bf16_splitk take (W, W_lo) as two bf16 operand streams into one fp32 accumulation. */
int prl_bf16_residual(const float* master, int64_t n, void* const* lo_dsts, int32_t n_dst, prl_stream_t stream);

/* Learner data parallelism as one fused exchange step over NVLink peer memory (replaces the gradient all-reduce
 * + per-rank full optimizer of finetune_loop.py:716-755): rank r owns elements [shard_begin, shard_end) of the
 * arena and ONLY that shard of fp32 master / exp_avg / exp_avg_sq (optimizer state sharded n_peers ways).
 *   prl_adamw_sharded_reduce : gsum = sum_p grads[p][shard] (P2P loads, fixed order), partial sum of squares
 *                              published into every rank's norm table (slot = rank).
 *   -- host barrier (all ranks reduced) --
 *   prl_adamw_sharded_update : clip by the global norm, AdamW on the shard, bf16 re-cast stored into EVERY rank's
 *                              parameter arena shadows[p][shard] (P2P stores).
 *   -- host barrier (all shards written) --
 * grads[]/shadows[]/norm_tables[] are the n_peers ranks' buffers in rank order (own and peers', mapped with
 * prl_ipc_open); norm_tables[p] is a double[n_peers] in rank p's memory. */
typedef struct {
  int64_t n, shard_begin, shard_end;
  float* master; float* exp_avg; float* exp_avg_sq;   /* [shard_end - shard_begin] */
  const void* grads[8];
  void* shadows[8];
  double* norm_tables[8];
  int32_t n_peers, rank, grad_is_bf16;
  float* gsum_scratch;                                /* [shard_end - shard_begin] fp32 */
  const int64_t* tensor_offsets; const uint8_t* tensor_no_decay; int32_t n_tensors;
  double lr, beta1, beta2, eps, weight_decay;
  int32_t step;
  float max_grad_norm, grad_scale;
} prl_adamw_shard_args;
int prl_adamw_sharded_reduce(const prl_adamw_shard_args* args, void* workspace, size_t workspace_bytes,
                             prl_stream_t stream);
int prl_adamw_sharded_update(const prl_adamw_shard_args* args, float* grad_norm_out, prl_stream_t stream);

/* ======================================================================= *
 * Feeder of hot path (2), GPU-resident (SURVEY §8 f1): one packed micro-batch row built on the learner's GPU from a
 * compact binary record (pipelinerl_b200/records.py) -- replaces populate_rl_data's pandas pipeline
 * (pipelinerl/finetune/rl/__init__.py:453-570), collate_packed's list -> tensor building (finetune/data.py:215-283)
 * and the JSONL round trip of the twelve [1, T] columns (streams.py:269-277, finetune_loop.py:109).
 * All pointers are DEVICE pointers into the uploaded record.  The `chunk` is the set of whole rollout groups the
 * statistics are taken over (preprocess.py:145-189: chunk_n_groups groups); the `pack` is the subset of its samples
 * that forms this micro-batch, in row order.  Float columns are double -> float roundings of exactly the doubles the
 * reference computes (Kahan sum / Welford std of pandas' groupby, rows in dataset order).
 * ======================================================================= */
typedef struct {
  int32_t n_chunk, n_pack, padding /* pad-to-seq_parallel sentinel tokens */, total_tok, total_lp;
  int32_t n_stat_slots, n_rollout_slots, n_groups;
  const double* reward;          /* [n_chunk] */
  const int32_t* stat_slot;      /* [n_chunk] dense id of (group_id, step_index) */
  const int32_t* rollout_slot;   /* [n_chunk] dense id of (group_id, rollout_index) */
  const int32_t* group_slot;     /* [n_chunk] dense id of group_id */
  const int32_t* n_tok_all;      /* [n_chunk] tokens of every chunk sample */
  const int32_t* pack_idx;       /* [n_pack] chunk index of each packed sample */
  const int32_t* pack_flags;     /* [n_pack] bit0 finished, bits1-2 finish_reason: 1 length, 2 stop|content_filter */
  const int32_t* tok_off;        /* [n_pack+1] */
  const int32_t* lp_off;         /* [n_pack+1] */
  const int32_t* input_ids;      /* [total_tok] packed samples, row order */
  const int32_t* labels;         /* [total_tok] */
  const float* logprobs;         /* [total_lp] sampler logprobs of the labelled tokens */
  const float* ref_logprobs;     /* [total_lp] or NULL (= logprobs: kl_coef == 0, preprocess.py:160-161) */
} prl_mb_record;
typedef struct {                 /* PipelineBatchEncoding columns, [1, total_tok + padding] each (types.py:46-180) */
  int64_t* input_ids; int64_t* labels; int64_t* attention_mask; int64_t* position_ids; int64_t* segment_ids;
  float* rewards; float* advantages; float* ref_logprobs; float* old_logprobs; float* group_tokens;
  float* num_labels; float* overflow;
  int32_t* seq_boundaries;       /* [n_pack + 1 (+1 with padding)] */
} prl_mb_columns;
size_t prl_preprocess_workspace_bytes(int32_t n_pack, int32_t n_stat_slots, int32_t n_rollout_slots, int32_t n_groups);
int prl_preprocess_pack(const prl_mb_record* record, int32_t divide_advantage_by_std, int32_t eos_token_id,
                        const prl_mb_columns* out, void* workspace, size_t workspace_bytes, prl_stream_t stream);

/* ======================================================================= *
 * Hot path (1): tcgen05 weight-streaming GEMM of the token step
 *   Y[M, N] = X[M, K] * W[N, K]^T, bf16 operands (row-major, K contiguous),
 *   fp32 accumulation in TMEM.  Replaces the cuBLAS GEMMs the vLLM engine runs
 *   per decode step for the reference (pipelinerl/async_llm.py:134 ->
 *   /v1/chat/completions; flags conf/base.yaml:59-73) and, with W_lo, the fp32
 *   lm_head matmul of pipelinerl/vllm_quantization.py:266-278
 *   (W_fp32 = W + W_lo with both parts bf16).
 *   Output: fp32 partial sums partials[split_k][M][N]; the consumer adds the
 *   splits in index order (deterministic).  K %% 8 == 0; pointers 16-B aligned.
 * ======================================================================= */
int prl_gemm_auto_split_k(int64_t M, int64_t N, int64_t K);
/* Tuning knob: shared-memory tile ring per CTA in KB (<= 100 lets two CTAs share an SM). */
int prl_gemm_set_smem_budget_kb(int32_t kb);
/* Weight layout switch: 0 = row-major [N,K]; 1 = contiguous 16 KB tiles [N/128][K/64][128][64] (one sequential
 * TMA box per tile; needs N % 128 == 0, K % 64 == 0). */
int prl_gemm_set_tiled_weights(int32_t on);
/* M_tok > 128 (chunked prefill / scoring / learner shapes): 1 (default) = CTA-pair kernel, one
 * tcgen05.mma.cta_group::2 256x256 tile per (2,1,1) cluster; 0 = the single-CTA 128x256 kernel. */
int prl_gemm_set_cta_pair(int32_t on);
/* Compute-bound GEMM of the learner body / prefill (csrc/gemm_tn.cu), replaces the cuBLAS GEMMs under the HF
 * Qwen2 forward+backward that rl_step drives (pipelinerl/finetune/rl/__init__.py:190-207, finetune_loop.py:716-725):
 *     C[M,N] (=|+=) alpha * A[M,K] * B[N,K]^T (+ bias[N]) (+ residual[M,N])
 * A, B bf16 row-major with row strides lda / ldb (elements, multiples of 8, base 16-byte aligned); C bf16 or fp32
 * (c_is_f32), `accumulate` (fp32 only) adds into C; bias / residual bf16 or NULL.  Persistent CTA-pair kernel
 * (tcgen05.mma.cta_group::2, 256x256 tiles, double-buffered TMEM accumulators). */
int prl_gemm_tn(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N, int64_t K,
                void* C, int64_t ldc, int32_t c_is_f32, int32_t accumulate, const void* bias,
                const void* residual, int64_t ldr, float alpha, prl_stream_t stream);
/* =======================================================================
 * Row-wise kernels of the learner body (csrc/learner_ops.cu): what HF's Qwen2RMSNorm / apply_rotary_pos_emb /
 * Qwen2MLP activation / embedding and their autograd backward do between the GEMMs of rl_step's model call
 * (pipelinerl/finetune/rl/__init__.py:190-207; backward finetune_loop.py:716-725).  bf16 activations [T, H]
 * contiguous unless a row stride is given; fp32 statistics; gradient reductions over tokens ACCUMULATE into fp32
 * outputs in a fixed order (workspace: prl_rowops_workspace_bytes(row length)).
 * ======================================================================= */
size_t prl_rowops_workspace_bytes(int64_t cols);
int prl_rmsnorm_fwd(const void* x, const void* gamma, int64_t T, int64_t H, float eps, void* y, float* rstd /*[T]*/,
                    prl_stream_t stream);
/* dx = (dres or 0) + dRMSNorm(x; gamma, rstd)(dy);  dgamma[H] += sum_t dy * x * rstd */
int prl_rmsnorm_bwd(const void* x, const void* gamma, const float* rstd, const void* dy, const void* dres /*or NULL*/,
                    int64_t T, int64_t H, void* dx, float* dgamma, void* workspace, size_t workspace_bytes,
                    prl_stream_t stream);
/* out[cols] += column sums of x [T, cols] (row stride ld): bias gradient */
int prl_colsum_bf16(const void* x, int64_t ld, int64_t T, int64_t cols, float* out, void* workspace,
                    size_t workspace_bytes, prl_stream_t stream);
/* rotate heads [0, n_heads) of every row of x [T, ld] in place by sign * pos[t] * inv_freq[i] (pairs (i, i + d/2));
 * sign = +1 forward, -1 backward (the transpose of a rotation) */
int prl_rope_inplace(void* x, int64_t ld, int64_t T, int32_t n_heads, int32_t head_dim, const int32_t* pos,
                     const float* inv_freq /*[head_dim/2]*/, float sign, prl_stream_t stream);
/* gate_up [T, 2I] = [gate | up] -> act [T, I] = silu(gate) * up, and its backward */
int prl_silu_mul_fwd(const void* gate_up, int64_t T, int64_t I, void* act, prl_stream_t stream);
int prl_silu_mul_bwd(const void* gate_up, const void* dact, int64_t T, int64_t I, void* dgate_up, prl_stream_t stream);
int prl_embed_gather(const void* table, const int64_t* ids, int64_t T, int64_t H, void* out, prl_stream_t stream);
/* dtable[ids[t]] += dh[t] (fp32 atomics: the one reduction here whose order is not fixed, as in torch) */
int prl_embed_scatter_add(float* dtable, const int64_t* ids, const void* dh, int64_t T, int64_t H, prl_stream_t stream);

/* Same kernel with either operand stored MN-major: a_mn_major -> A is given as [K, M] row-major (row stride lda >= M),
 * b_mn_major -> B as [K, N] row-major.  dgrad (dX = dY W, B = W as stored) and wgrad (dW += dY^T X, both operands as
 * stored) need no transposed copies this way. */
int prl_gemm_ex(const void* A, int64_t lda, int32_t a_mn_major, const void* B, int64_t ldb, int32_t b_mn_major,
                int64_t M, int64_t N, int64_t K, void* C, int64_t ldc, int32_t c_is_f32, int32_t accumulate,
                const void* bias, const void* residual, int64_t ldr, float alpha, prl_stream_t stream);
/* gate_up GEMM with SwiGLU in its epilogue (the MLP of the HF block the reference runs, rl/__init__.py:190-207):
 * act[M, I] = silu(X Wg^T) * (X Wu^T) with W = [Wg; Wu] ([2 I, K], as gate_up_proj is stored); the two CTAs of a pair stage
 * the gate rows and the up rows of the same 128 features, so one accumulator row holds both halves and the activation
 * never makes a round trip through HBM.  gate_up ([M, 2 I] bf16) is written too when non-NULL (kept for the backward).
 * Bit-identical to prl_gemm_ex + prl_silu_mul_fwd.  I must be a multiple of 128. */
int prl_gemm_swiglu(const void* X, int64_t ldx, const void* W, int64_t ldw, int64_t M, int64_t I, int64_t K, void* act,
                    int64_t ld_act, void* gate_up /*or NULL*/, int64_t ld_gate_up, prl_stream_t stream);
/* sampler form (chunked prefill): act = bf16(SiLU(gate) * up) of the fp32 accumulators, i.e. the bits of
 * prl_gemm_tn(fp32 out) + prl_silu_mul without the [M, 2I] fp32 round trip through HBM */
int prl_gemm_swiglu_f32(const void* X_bf16, int64_t ldx, const void* W_gate_up_bf16, int64_t ldw, int64_t M, int64_t I,
                        int64_t K, void* act_bf16, int64_t ld_act, prl_stream_t stream);
/* down_proj dgrad with the backward of SiLU(gate) * up in its epilogue: d_gate_up[M, 2 I] (= d gate | d up) from dY[M, H],
 * W_down[H, I] as stored and the forward's gate_up[M, 2 I]; d act is never written.  Bit-identical to
 * prl_gemm_ex(dY, W_down as MN-major B) followed by prl_silu_mul_bwd.  Needs I % 32 == 0. */
int prl_gemm_dgrad_swiglu(const void* dY_bf16, int64_t ldy, const void* W_down_bf16, int64_t ldw, int64_t M, int64_t I, int64_t H,
                          const void* gate_up_bf16, void* d_gate_up_bf16, int64_t ld_gu, prl_stream_t stream);
/* bf16 [rows, cols] (row stride ld_in) -> [cols, rows] (row stride ld_out): stages the K-major operands of wgrad. */
int prl_transpose_bf16(const void* in, int64_t rows, int64_t cols, int64_t ld_in, void* out, int64_t ld_out,
                       prl_stream_t stream);
int prl_gemm_bf16_splitk(const void* W, const void* W_lo /*or NULL*/, const void* X,
                         int64_t M, int64_t N, int64_t K, int32_t split_k /*0 = auto*/,
                         float* partials, prl_stream_t stream);
/* Token-step gate_up GEMM with SiLU(gate) * up in its epilogue (M <= 128 tokens, split_k = 1): act[M, I] bf16 = the bits
 * of prl_gemm_bf16_splitk(split_k = 1) followed by prl_silu_mul, in one launch (vLLM: fused SiluAndMul after the
 * gate_up_proj GEMM).  W = gate_up_proj.weight [2 I, K] as stored, gate rows first. */
int prl_gemm_swiglu_decode(const void* W_bf16, const void* X_bf16, int64_t M, int64_t I, int64_t K, void* act_bf16,
                           prl_stream_t stream);

/* Fused output head with IN-KERNEL logprob capture: logits = X W^T (+ W_lo) are produced tile by tile in
 * TMEM and reduced on the spot — per token logsumexp, exact entropy, the log-probability of a given target
 * (teacher forcing: the trainer's new_logprobs, rl/__init__.py:207-233, and the reference-logprob scoring of
 * llm.py:606-648) and/or a sample from softmax(logits/T) with its log-probability (the sampler +
 * processed_logprobs path, conf/base.yaml:65).  Full-vocabulary logits (608 KB/token in fp32 for Qwen2.5)
 * never reach HBM.  Any output pointer may be NULL.  Sampling uses the same counter-based RNG as
 * prl_sample_logprob (row = token index). */
size_t prl_head_workspace_bytes(int64_t M, int64_t V);
int prl_head_logprob(const void* W /*[V,K] bf16*/, const void* W_lo /*or NULL*/, const void* X /*[M,K] bf16*/,
                     int64_t M, int64_t V, int64_t K, float temperature, const int64_t* targets /*[M] or NULL*/,
                     int32_t greedy, uint64_t seed, uint32_t step, float* logprob_target, float* entropy, float* lse,
                     int32_t* sampled_ids, float* sampled_logprobs, void* workspace, size_t workspace_bytes,
                     prl_stream_t stream);

/* ======================================================================= *
 * Hot path (1): fused epilogue kernels of one token step and paged attention.
 *   Together with prl_gemm_bf16_splitk these are the decode step the
 *   reference delegates to the vLLM engine (client: pipelinerl/async_llm.py:86-212;
 *   server flags conf/base.yaml:59-73; fp32 head vllm_quantization.py:128-278):
 *   fused_add_rms_norm, rotary_embedding, reshape_and_cache, paged attention,
 *   silu_and_mul, sampler + processed_logprobs.
 *   All activations: one row per token; `partials` are GEMM split-K partials
 *   [n_split][B][cols] fp32.  KV cache (bf16), page_size 64, head_dim 128:
 *     row(layer, kv, page, kvh, slot) = (((layer*2+kv)*n_pages + page)*n_kv + kvh)*64 + slot
 * ======================================================================= */
int prl_embed_rmsnorm(const int32_t* tokens, const void* embed_bf16, const void* gamma_bf16, float eps,
                      int32_t B, int32_t H, int32_t vocab, float* h /*[B,H] residual, out*/,
                      void* x_bf16 /*[B,H] out*/, prl_stream_t stream);
/* `l2_prefetch` (nullable) on the three epilogue kernels below: a weight range of an UPCOMING GEMM to pull into
 * the 126 MB L2 (evict_last) while the long HBM-bound kernel that runs in between hides the DRAM latency. */
int prl_residual_rmsnorm(const float* partials, int32_t n_split, int32_t B, int32_t H, const void* gamma_bf16,
                         float eps, float* h /*in/out*/, void* x_bf16 /*out*/, const void* l2_prefetch,
                         size_t l2_prefetch_bytes, prl_stream_t stream);
int prl_qkv_rope_cache(const float* partials, int32_t n_split, int32_t B, const void* bias_bf16 /*or NULL*/,
                       int32_t n_q, int32_t n_kv, int32_t head_dim, const int32_t* positions /*[B]*/,
                       const int32_t* block_table /*[slots,max_blocks]*/, int32_t max_blocks,
                       const int32_t* row_slot /*[B] block-table row of each token row, or NULL = identity*/,
                       const float* inv_freq /*[head_dim/2]*/, void* q_out_bf16 /*[B,n_q,128]*/,
                       void* kv_cache_bf16, int64_t n_pages, int32_t layer, int32_t page_size,
                       const void* l2_prefetch, size_t l2_prefetch_bytes, prl_stream_t stream);
int prl_silu_mul(const float* partials, int32_t n_split, int32_t B, int32_t I, void* act_bf16 /*[B,I]*/,
                 const void* l2_prefetch, size_t l2_prefetch_bytes, prl_stream_t stream);
int prl_paged_attn_splits(int32_t B, int32_t n_kv, int32_t max_seq_len);
/* The workspace must be zero-filled once before its first use (arrival counters; they re-arm themselves). */
size_t prl_paged_attn_workspace_bytes(int32_t B, int32_t n_q, int32_t n_splits);
int prl_paged_attn_decode(const void* q_bf16, const void* kv_cache_bf16, int64_t n_pages, int32_t n_layers,
                          int32_t layer, const int32_t* block_table, int32_t max_blocks,
                          const int32_t* seq_lens /*[B] tokens in cache incl. the current one*/,
                          int32_t B, int32_t n_q, int32_t n_kv, int32_t head_dim, int32_t page_size,
                          int32_t n_splits, float sm_scale, void* out_bf16 /*[B, n_q*128]*/,
                          void* workspace, size_t workspace_bytes, prl_stream_t stream);
/* Chunked prefill: causal attention of seq_q_len[z] query rows (starting at row seq_q_start[z], first
 * position seq_pos0[z]) against the paged KV of block-table row seq_slot[z]; the chunk's own K/V must
 * already be in the cache (prl_qkv_rope_cache).  Replaces vLLM's chunked-prefill attention
 * (conf/base.yaml:64,72). */
int prl_paged_attn_prefill(const void* q_bf16 /*[rows,n_q,128]*/, const void* kv_cache_bf16, int64_t n_pages,
                           int32_t n_layers, int32_t layer, const int32_t* block_table, int32_t max_blocks,
                           const int32_t* seq_q_start, const int32_t* seq_q_len, const int32_t* seq_pos0,
                           const int32_t* seq_slot, int32_t n_seqs, int32_t max_q_len, int32_t n_q, int32_t n_kv,
                           int32_t head_dim, int32_t page_size, float sm_scale, void* out_bf16 /*[rows,n_q*128]*/,
                           prl_stream_t stream);
/* Same contract on the tcgen05 path (csrc/attn_tc.cu): a query tile packs 128 / (n_q / n_kv) tokens x the GQA group's
 * heads into one UMMA tile, S = Q K^T and P V run on the tensor core with TMEM accumulators, V is read as stored
 * (MN-major operand).  q_rows = rows of the q buffer that hold this chunk (TMA bounds). */
int prl_paged_attn_prefill_tc(const void* q_bf16 /*[q_rows,n_q,128]*/, int32_t q_rows, const void* kv_cache_bf16,
                              int64_t n_pages, int32_t n_layers, int32_t layer, const int32_t* block_table,
                              int32_t max_blocks, const int32_t* seq_q_start, const int32_t* seq_q_len,
                              const int32_t* seq_pos0, const int32_t* seq_slot, int32_t n_seqs, int32_t max_q_len,
                              int32_t n_q, int32_t n_kv, int32_t head_dim, int32_t page_size, float sm_scale,
                              void* out_bf16 /*[rows,n_q*128]*/, prl_stream_t stream);
/* Learner attention (hot path 2): block-diagonal causal attention over ONE packed row and its backward -- the
 * flash-attn varlen call the reference makes through HF with packed position_ids
 * (pipelinerl/finetune/rl/__init__.py:204 forward, finetune_loop.py:716-725 backward; conf/finetune/base.yaml:12-13,64).
 * qkv: [T, qkv_stride] bf16 rows = [n_q q heads | n_kv k heads | n_kv v heads] x 128, q / k already roped.
 * Segment z = rows [seg_start[z], seg_start[z] + seg_len[z]); head_dim must be 128, n_q / n_kv <= 64.
 * fwd: out [T, n_q*128] bf16, lse [T, n_q] fp32 (log2 domain of the scaled scores; NULL = not needed).
 * bwd: dqkv [T, dqkv_stride] bf16 in the layout of qkv (every segment row is written); dK / dV are reduced over
 * the GQA group inside the tensor core in a fixed order (deterministic, no atomics).
 * csrc/attn_tc.cu (forward) and csrc/attn_train.cu (backward): tcgen05 MMAs, TMEM accumulators, TMA operands. */
int prl_attn_varlen_fwd(const void* qkv_bf16, int64_t qkv_stride, int32_t T, const int32_t* seg_start,
                        const int32_t* seg_len, int32_t n_seg, int32_t max_seg_len, int32_t n_q, int32_t n_kv,
                        int32_t head_dim, float sm_scale, void* out_bf16, float* lse, prl_stream_t stream);
/* which forward kernel prl_attn_varlen_fwd launches: 2 (default) = two ping-pong softmax groups, O accumulated in TMEM
 * with conditional rescale; 1 = the first-generation kernel shared with chunked prefill.  For A/B runs and tests. */
int prl_attn_set_fwd_generation(int32_t generation);
/* same switch for prl_paged_attn_prefill_tc (chunked prefill / scoring): default 2 */
int prl_attn_set_prefill_generation(int32_t generation);
/* backward kernels: 2 (default) = P^T / dS^T / dS reach the tensor core through TMEM (A operand in tensor memory);
 * 1 = through shared memory.  For A/B runs and tests. */
int prl_attn_set_bwd_generation(int32_t generation);
size_t prl_attn_varlen_bwd_workspace_bytes(int32_t T, int32_t n_q);
int prl_attn_varlen_bwd(const void* qkv_bf16, int64_t qkv_stride, int32_t T, const int32_t* seg_start,
                        const int32_t* seg_len, int32_t n_seg, int32_t max_seg_len, int32_t n_q, int32_t n_kv,
                        int32_t head_dim, float sm_scale, const void* out_bf16, const void* d_out_bf16,
                        const float* lse, void* dqkv_bf16, int64_t dqkv_stride, void* workspace,
                        size_t workspace_bytes, prl_stream_t stream);
/* Sequence-parallel forms (the reference shards a packed row over `seq_parallel` ranks and runs ring attention:
 * finetune_loop.py:507-517,757-759, finetune/types.py:145-180).  The queries are the LOCAL slice q[Tq, q_stride] (query heads
 * in the first n_q * 128 columns -- the local qkv matrix qualifies), the keys / values the all-gathered
 * kv[Tkv, kv_stride] = [k heads | v heads].  Local segment z = q rows [seg_q_start[z], + seg_q_len[z]); its first query
 * sits at position seg_pos0[z] of its sequence, whose first key is kv row seg_kv_start[z].  The backward writes the local
 * dq[Tq, dq_stride] and THIS RANK'S contribution dkv[Tkv, dkv_stride] = [dK | dV] to every key row (zero where no local
 * query attends); the caller reduce-scatters dkv over the group. */
int prl_attn_varlen_fwd_kv(const void* q_bf16, int64_t q_stride, int32_t Tq, const void* kv_bf16, int64_t kv_stride,
                           int32_t Tkv, const int32_t* seg_q_start, const int32_t* seg_q_len, const int32_t* seg_pos0,
                           const int32_t* seg_kv_start, int32_t n_seg, int32_t max_q_len, int32_t n_q, int32_t n_kv,
                           int32_t head_dim, float sm_scale, void* out_bf16, float* lse, prl_stream_t stream);
int prl_attn_varlen_bwd_kv(const void* q_bf16, int64_t q_stride, int32_t Tq, const void* kv_bf16, int64_t kv_stride,
                           int32_t Tkv, const int32_t* seg_q_start, const int32_t* seg_q_len, const int32_t* seg_pos0,
                           const int32_t* seg_kv_start, int32_t n_seg, int32_t max_q_len, int32_t max_kv_len,
                           int32_t n_q, int32_t n_kv, int32_t head_dim, float sm_scale, const void* out_bf16,
                           const void* d_out_bf16, const float* lse, void* dq_bf16, int64_t dq_stride, void* dkv_bf16,
                           int64_t dkv_stride, void* workspace, size_t workspace_bytes, prl_stream_t stream);
/* Measurement helper (tools/attn_bench.py --tmem): cycles for `warps` warps of every SM to read iters x 4 KB out of
 * TMEM with tcgen05.ld.32x32b.x32; out3 = {cycles, bytes per SM, -}. */
int prl_debug_tmem_read_bench(int32_t iters, int32_t warps, int64_t* out3_device, prl_stream_t stream);
/* measurement helper: tcgen05.mma throughput per operand configuration (modes 0-9, batches of 8 UMMAs under one lane
 * election) and the softmax <-> tensor-core hand-off round trip (mode 10); out2_device[0] = cycles, [1] = UMMAs issued
 * (profiles/r2_attention.md) */
/* measurement helper: per-phase cycle sums of one CTA of the generation-2 learner attention forward (20 int64; NULL = off) */
int prl_attn_debug_timing(int64_t* out20_device);
/* likewise for the generation-4 dQ backward kernel (16 int64; NULL = off) */
int prl_attn_debug_bwd_timing(int64_t* out16_device);
int prl_attn_debug_bwd_timing_dkdv(int64_t* out16_device);
int prl_debug_mma_bench(int32_t mode, int32_t iters, int64_t* out2_device, prl_stream_t stream);
/* Sampling with in-kernel logprob capture: id ~ softmax(logits/T) (Gumbel-max, counter-based RNG on
 * (seed, step, row, vocab id)) or argmax when greedy; logprob = log_softmax(logits/T)[id]. */
size_t prl_sample_workspace_bytes(int32_t B);
int prl_sample_logprob(const float* logits /*[B,V]*/, int32_t B, int32_t V, float temperature, int32_t greedy,
                       uint64_t seed, uint32_t step, int32_t* out_ids, float* out_logprobs,
                       void* workspace, size_t workspace_bytes, prl_stream_t stream);
/* Same with PER-SEQUENCE sampling parameters (inv_temperature_rows[b] = 1 / T_b, greedy_rows[b]): requests admitted with
 * different `llm.parameters` (train handle at T = 1, eval handle greedy ...) share one engine batch, and every sequence's
 * logprobs stay those of ITS OWN distribution (what rl_step assumes via RLConfig.temperature). */
int prl_sample_logprob_rows(const float* logits /*[B,V]*/, int32_t B, int32_t V, const float* inv_temperature_rows,
                            const uint8_t* greedy_rows, uint64_t seed, uint32_t step, int32_t* out_ids,
                            float* out_logprobs, void* workspace, size_t workspace_bytes, prl_stream_t stream);
/* top-k / top-p filtering with processed logprobs (vLLM's apply_top_k_top_p + log_softmax of the masked logits).
 * Call after prl_sample_logprob_rows with the same logits, seed and step.  For every row that is not greedy and has an
 * active filter (1 <= top_k_rows[b] < V, or top_p_rows[b] < 1) it rewrites out_ids[b] / out_logprobs[b]: the kept set
 * is {z >= tau}, z = logits[b] * inv_temperature_rows[b], with tau the k-th largest z and then the value where the
 * softmax mass of the survivors ranked strictly above reaches top_p (every tie with tau is kept); the id is the
 * Gumbel-max over the kept set with prl_sample_logprob_rows' noise (an unfiltered sample inside the kept set is kept
 * as is) and the logprob is z[id] - logsumexp(z over the kept set).  Other rows are left untouched.
 * top_k_rows[b] in {-1, 0} or >= V disables top-k; top_p_rows[b] == 1 disables top-p.  The per-row values live in
 * device memory, so they are checked on the device: a row with top_p outside (0, 1] or top_k < -1 keeps its
 * unfiltered sample and reports out_kept[b] = -1.  out_kept[b] (optional) is the kept-set size, V for unfiltered rows.
 * Deterministic: the same inputs give the same bits. */
size_t prl_sample_filter_workspace_bytes(int32_t B, int32_t V);
int prl_sample_filter_rows(const float* logits /*[B,V]*/, int32_t B, int32_t V, const float* inv_temperature_rows,
                           const uint8_t* greedy_rows, const int32_t* top_k_rows, const float* top_p_rows,
                           uint64_t seed, uint32_t step, int32_t* out_ids, float* out_logprobs,
                           int32_t* out_kept /*[B] kept-set size, or NULL*/, void* workspace, size_t workspace_bytes,
                           prl_stream_t stream);
/* Device-resident scheduler state of one sampler (all pointers device, one entry per slot).
 * prl_advance_state moves every active slot one token forward without a host round trip:
 * feeds the next prompt token while inside the prompt, else appends (sampled id, logprob) to the
 * slot's output ring, and retires the slot on EOS (finished=1, "stop") or max_new (finished=2, "length")
 * — the finish_reason values pipelinerl/async_llm.py:202-212 reports. */
typedef struct {
  int32_t B;
  const int32_t* sampled;          /* [B] ids drawn by prl_sample_logprob this step */
  const float* sampled_logprobs;   /* [B] */
  int32_t* tokens;                 /* [B] next input token (in/out) */
  int32_t* positions;              /* [B] position of `tokens` */
  int32_t* seq_lens;               /* [B] tokens in the KV cache incl. the current one; 0 = slot idle */
  uint8_t* active;                 /* [B] */
  const int32_t* prompt_buf;       /* [B, prompt_stride] */
  int32_t prompt_stride;
  const int32_t* prompt_len;       /* [B] */
  int32_t* out_ids;                /* [B, out_stride] */
  float* out_logprobs;             /* [B, out_stride] */
  int32_t out_stride;
  int32_t* gen_count;              /* [B] */
  const int32_t* max_new;          /* [B] */
  uint8_t* finished;               /* [B] 0 running, 1 stop, 2 length */
  int32_t eos_id;
  int32_t ignore_eos;              /* engine-wide: never stop on eos */
  const uint8_t* ignore_eos_rows;  /* [B] per sequence (may be NULL) */
} prl_engine_state;
int prl_advance_state(const prl_engine_state* state, prl_stream_t stream);

/* ---- tensor parallelism inside one engine (BASELINE config 4: Qwen2.5-32B, TP=2; the reference passes
 * tensor-parallel-size to vLLM, world.py:56-59, which all-reduces twice per layer with NCCL/custom all-reduce).
 * Here the row-parallel GEMMs (o_proj, down_proj) store their fp32 partial tiles into the local AND the peer GPU's
 * reduction buffer in their epilogue (prl_gemm_bf16_splitk_peer: the all-reduce is fused into the GEMM over NVLink
 * peer memory); the consumer (prl_residual_rmsnorm) then reduces tp x split slots in a fixed order, so both ranks
 * compute bit-identical residual streams.  Ordering between the GPUs uses counters in peer memory:
 *   prl_tp_signal(peer counter)        after this rank's P2P stores (stream order + system fence)
 *   prl_tp_wait(local counter, epoch, signals_per_step, k)   before consuming the peer's k-th delivery of the step
 *   prl_tp_epoch(epoch)                once per token step.
 * The vocab-parallel head exchanges 16 sampler partials per row instead of logits (prl_sample_partials with a
 * vocabulary offset, prl_weights_push of the partials, prl_sample_finalize over both groups). */
int prl_gemm_bf16_splitk_peer(const void* W, const void* X, int64_t M, int64_t N, int64_t K, int32_t split_k,
                              float* partials, float* peer_partials, prl_stream_t stream);
int prl_tp_signal(void* peer_flag, prl_stream_t stream);
int prl_tp_wait(const void* flag, const void* epoch, int32_t signals_per_step, int32_t k, prl_stream_t stream);
int prl_tp_epoch(void* epoch, prl_stream_t stream);
int prl_sample_partials(const float* logits, int32_t B, int32_t V, float temperature, int32_t greedy, uint64_t seed,
                        uint32_t step, int32_t vocab_offset, void* partials /*[B][16] x 32 B*/, prl_stream_t stream);
int prl_sample_finalize(const void* partials /*[n_groups][B][16]*/, int32_t B, int32_t n_groups, int32_t* out_ids,
                        float* out_logprobs, prl_stream_t stream);

/* ======================================================================= *
 * Hot path (3): in-flight weight update as a one-shot NVLink P2P copy
 *   replaces WeightUpdateManager.send_weight_update (pipelinerl/finetune_loop.py:205-292),
 *   WorkerExtension.receive_weight_update (pipelinerl/vllm1.py:110-127) and the PyNccl group of
 *   pipelinerl/torch_utils.py:70-94.  Sampler side (once): allocate the two arena buffers and a
 *   16-byte control block with prl_ipc_alloc, export their handles.  Learner side: open the handles,
 *   then per update prl_weights_push (its byte slice -> every sampler's inactive buffer) followed by
 *   prl_weights_signal on the same stream.  Control block: u64 version (max of pushed versions),
 *   u64 arrivals (monotonic count of signals); the sampler flips buffers at a token-step boundary
 *   when arrivals has advanced by the number of pushing learner ranks.
 * ======================================================================= */
int prl_ipc_alloc(size_t bytes, void** dptr);
int prl_ipc_free(void* dptr);
int prl_ipc_export(const void* dptr, uint8_t handle[64]);
int prl_ipc_open(const uint8_t handle[64], void** dptr);
int prl_ipc_close(void* dptr);
int prl_enable_peer_access(int32_t peer_device);
int prl_weights_push(const void* src_arena, void* const* dst_arenas, int32_t n_dst, size_t offset_bytes,
                     size_t bytes, int32_t max_ctas /*0 = 2 per SM*/, prl_stream_t stream);
int prl_weights_signal(void* const* ctrl_blocks, int32_t n_dst, uint64_t version, prl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PRL_H_ */
