// Hot path (1), sampler: top-k / top-p filtering with processed logprobs.
//
// Replaces, for the reference's eval handle (`test_llm`: top_p 0.95, top_k 50, conf/base.yaml:52-57), vLLM's
// apply_top_k_top_p + log_softmax of the masked logits (logprobs-mode processed_logprobs, conf/base.yaml:65).
// For one row with z = logits * (1/T):
//   top-k (1 <= k < V):  tau_k = the k-th largest z; keep {z >= tau_k} (every tie with the k-th value is kept)
//   top-p (p < 1):       over the top-k survivors, keep a token iff the softmax mass of the tokens ranked strictly
//                        above it is < p of the survivors' mass; ties with the boundary value are all kept, so the
//                        kept set is always {z >= tau} (vLLM's unstable sort may split such a tie)
//   id      = argmax over the kept set of z + gumbel(seed, step, row, id)  (the noise of sample_partial_kernel: a row
//             whose unfiltered sample is kept draws the same token)
//   logprob = z[id] - logsumexp(z over the kept set)
//
// One CTA per row.  Thresholds come from a radix select on the order-preserving uint32 image of z, 8 bits per round
// (4 rounds), over shared-memory histograms of counts (top-k) or of counts and softmax mass (top-p).  The row is
// re-read from L2 (the sampler has just read it), until the candidates above the current bucket fit in shared memory:
// from then on every round and the final pass read the compacted candidates.  Masses are exp(z - max) in 2^-40
// fixed point, summed with integer atomics, so every threshold and the kept-set logsumexp are independent of the
// order in which threads add them: results are bitwise deterministic.
#include "prl_common.cuh"
#include <math.h>

namespace prl {
namespace {

constexpr int kFilterThreads = 1024;
constexpr int kFilterCap = 8192;                  // candidates compacted into shared memory (z and id: 64 KB)
constexpr int kFilterMaxVocab = 1 << 23;          // V * 2^40 must fit the uint64 mass sums
constexpr float kMassOne = 1099511627776.f;       // 2^40 = exp(0) in fixed point

__device__ __forceinline__ uint32_t order_key(float z) {
  const uint32_t u = __float_as_uint(z == 0.f ? 0.f : z);   // -0 and +0 compare equal: give them one key
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ unsigned long long fixed_mass(float z, float M) {
  return __float2ull_rn(__expf(z - M) * kMassOne);
}

struct Pick { float v; int i; };
__device__ __forceinline__ Pick better(Pick a, Pick b) {   // ties -> lowest index, as sample_partial_kernel
  if (b.v > a.v || (b.v == a.v && b.i < a.i)) return b;
  return a;
}

// Radix-select state, written by one lane of warp 0 between rounds and read by the whole CTA after a barrier.
struct Select {
  uint32_t prefix;                  // the `done` high bits of the threshold key chosen so far
  int done;                         // 0, 8, 16, 24, 32
  unsigned long long above_cnt;     // elements (within the restriction) above the current bucket
  unsigned long long above_mass;
  unsigned long long target;        // k (count select) or p * survivors' mass (mass select)
  unsigned long long n_cand;        // above_cnt + elements in the current bucket
};

struct FilterShared {
  uint32_t cnt[256];
  unsigned long long mass[256];
  Select sel;
  int n_smem;                       // compacted candidates; -1 while the row is read from global memory
  int n_fill;                       // compaction cursor
  float red_f[32];
  float red_v[32];
  int red_i[32];
  unsigned long long red_m[32];
};

// Visit every element of the row (z = logits * inv_temp, the sampler's fp32 multiply) as f(z, id): 4 float4 loads in
// flight per thread when the row is 16-byte aligned.
template <class F>
__device__ __forceinline__ void for_row(const float* __restrict__ row, int V, float inv_temp, F&& f) {
  int lo = 0;
  if ((reinterpret_cast<uintptr_t>(row) & 15) == 0) {
    constexpr int U = 4;
    const int V4 = V >> 2;
    const float4* r4 = reinterpret_cast<const float4*>(row);
    int i = threadIdx.x;
    for (; i + (U - 1) * kFilterThreads < V4; i += U * kFilterThreads) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = __ldcg(r4 + i + u * kFilterThreads);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int id = (i + u * kFilterThreads) * 4;
        f(v[u].x * inv_temp, id); f(v[u].y * inv_temp, id + 1); f(v[u].z * inv_temp, id + 2); f(v[u].w * inv_temp, id + 3);
      }
    }
    for (; i < V4; i += kFilterThreads) {
      const float4 v = __ldcg(r4 + i);
      const int id = i * 4;
      f(v.x * inv_temp, id); f(v.y * inv_temp, id + 1); f(v.z * inv_temp, id + 2); f(v.w * inv_temp, id + 3);
    }
    lo = V4 * 4;
  }
  for (int i = lo + threadIdx.x; i < V; i += kFilterThreads) f(__ldcg(row + i) * inv_temp, i);
}

// Warp 0: pick the bucket of the next 8 key bits that holds the threshold — the first bucket, from the top, where the
// running total (count, or mass when by_mass) reaches sel.target.  With target_p > 0 the target is first set to
// target_p times the total mass of this round (the survivors' mass: the first round of a mass select sees them all).
__device__ void choose_bucket(FilterShared& sh, bool by_mass, float target_p) {
  const int lane = threadIdx.x & 31;
  Select& s = sh.sel;
  unsigned long long c[8], m[8], csum = 0, msum = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int bin = 255 - (lane * 8 + j);
    c[j] = sh.cnt[bin];
    m[j] = sh.mass[bin];
    csum += c[j];
    msum += m[j];
  }
  unsigned long long cinc = csum, minc = msum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long ct = __shfl_up_sync(0xffffffffu, cinc, o), mt = __shfl_up_sync(0xffffffffu, minc, o);
    if (lane >= o) { cinc += ct; minc += mt; }
  }
  unsigned long long target = s.target;
  if (target_p > 0.f) {   // at least 1: the most likely token (mass 2^40) is always kept
    target = (unsigned long long)((double)__shfl_sync(0xffffffffu, minc, 31) * (double)target_p);
    if (target == 0) target = 1;
  }
  const unsigned long long base = by_mass ? s.above_mass : s.above_cnt;
  const unsigned hit = __ballot_sync(0xffffffffu, base + (by_mass ? minc : cinc) >= target);
  const unsigned nonempty = __ballot_sync(0xffffffffu, csum > 0);
  // no bucket reaches the target only if rounding left it above the total: then keep everything (the lowest bucket)
  const int first = hit ? __ffs(hit) - 1 : 31 - __clz(nonempty);
  if (lane == first) {
    unsigned long long ac = s.above_cnt + (cinc - csum), am = s.above_mass + (minc - msum);
    int j = 0;
    if (hit) {
      while (j < 7 && (by_mass ? am + m[j] : ac + c[j]) < target) { ac += c[j]; am += m[j]; ++j; }
    } else {
      int last = 7;
      while (last > 0 && c[last] == 0) --last;
      for (; j < last; ++j) { ac += c[j]; am += m[j]; }
    }
    s.prefix = (s.done ? s.prefix << 8 : 0u) | (uint32_t)(255 - (lane * 8 + j));
    s.done += 8;
    s.above_cnt = ac;
    s.above_mass = am;
    s.n_cand = ac + c[j];
    s.target = target;
  }
}

__global__ void __launch_bounds__(kFilterThreads, 1) sample_filter_kernel(
    const float* __restrict__ logits, int V, const float* __restrict__ inv_temp_rows,
    const uint8_t* __restrict__ greedy_rows, const int32_t* __restrict__ top_k_rows,
    const float* __restrict__ top_p_rows, uint64_t seed, uint32_t step, int32_t* __restrict__ out_ids,
    float* __restrict__ out_logprobs, int32_t* __restrict__ out_kept) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ FilterShared sh;
  extern __shared__ float s_dyn[];
  float* s_z = s_dyn;
  int* s_id = reinterpret_cast<int*>(s_dyn + kFilterCap);
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int k = top_k_rows[b];
  const float p = top_p_rows[b];
  if (!(p > 0.f && p <= 1.f) || k < -1) {           // invalid row: the unfiltered sample stands, out_kept flags it
    if (out_kept && tid == 0) out_kept[b] = -1;
    return;
  }
  const bool use_k = k >= 1 && k < V, use_p = p < 1.f;
  if (greedy_rows[b] || !(use_k || use_p)) {       // greedy ignores both filters (vLLM resets them below its eps)
    if (out_kept && tid == 0) out_kept[b] = V;
    return;
  }
  const float inv_temp = inv_temp_rows[b];
  const float* row = logits + (int64_t)b * V;

  // the candidates live in shared memory once sh.n_smem >= 0
  auto for_each = [&](auto&& f) {
    const int n = sh.n_smem;
    if (n >= 0) {
      for (int j = tid; j < n; j += kFilterThreads) f(s_z[j], s_id[j]);
    } else {
      for_row(row, V, inv_temp, f);
    }
  };
  auto clear_hist = [&]() {
    for (int i = tid; i < 256; i += kFilterThreads) { sh.cnt[i] = 0u; sh.mass[i] = 0ull; }
  };

  // ---- pass 0: max; the first top-k round; compaction when the whole row fits ----
  if (tid == 0) {
    sh.n_smem = -1;
    sh.n_fill = 0;
    sh.sel = Select{0u, 0, 0ull, 0ull, (unsigned long long)(use_k ? k : 0), (unsigned long long)V};
  }
  clear_hist();
  __syncthreads();
  float M = -INFINITY;
  {
    const bool compact = V <= kFilterCap;
    int run_bin = -1;
    uint32_t run_cnt = 0;
    for_each([&](float z, int id) {
      M = fmaxf(M, z);
      if (compact) {
        const int pos = atomicAdd(&sh.n_fill, 1);
        s_z[pos] = z;
        s_id[pos] = id;
      }
      if (use_k) {
        const int bin = (int)(order_key(z) >> 24);
        if (bin != run_bin) {
          if (run_cnt) atomicAdd(&sh.cnt[run_bin], run_cnt);
          run_bin = bin;
          run_cnt = 0;
        }
        ++run_cnt;
      }
    });
    if (run_cnt) atomicAdd(&sh.cnt[run_bin], run_cnt);
    M = warp_max(M);
    if (lane == 0) sh.red_f[warp] = M;
    __syncthreads();
    M = sh.red_f[0];
    for (int w = 1; w < kFilterThreads / 32; ++w) M = fmaxf(M, sh.red_f[w]);
    if (compact && tid == 0) sh.n_smem = sh.n_fill;
  }

  // One radix round over the candidates with key >= lo_key whose high bits equal the chosen prefix: histogram of the
  // next 8 bits (count, plus mass for a mass select), compacting the candidates of the current bucket and above into
  // shared memory on the way when they fit.  Each thread adds runs of equal buckets at once (neighbouring logits of
  // one row mostly share the high bits), which keeps shared atomics off the critical path.
  auto round = [&](bool by_mass, uint32_t lo_key) {
    const Select s = sh.sel;
    const bool compact = sh.n_smem < 0 && s.n_cand <= (unsigned long long)kFilterCap;
    const uint32_t bucket_lo = s.done ? (s.prefix << (32 - s.done)) : 0u;
    const uint32_t cand_lo = bucket_lo > lo_key ? bucket_lo : lo_key;
    const int shift = 24 - s.done;
    int run_bin = -1;
    uint32_t run_cnt = 0;
    unsigned long long run_mass = 0;
    for_each([&](float z, int id) {
      const uint32_t key = order_key(z);
      if (key < cand_lo) return;
      if (compact) {
        const int pos = atomicAdd(&sh.n_fill, 1);
        if (pos < kFilterCap) { s_z[pos] = z; s_id[pos] = id; }
      }
      if (s.done && (key >> (32 - s.done)) != s.prefix) return;
      const int bin = (int)((key >> shift) & 255u);
      if (bin != run_bin) {
        if (run_cnt) { atomicAdd(&sh.cnt[run_bin], run_cnt); atomicAdd(&sh.mass[run_bin], run_mass); }
        run_bin = bin;
        run_cnt = 0;
        run_mass = 0;
      }
      ++run_cnt;
      if (by_mass) run_mass += fixed_mass(z, M);
    });
    if (run_cnt) { atomicAdd(&sh.cnt[run_bin], run_cnt); atomicAdd(&sh.mass[run_bin], run_mass); }
    __syncthreads();
    if (compact && tid == 0) sh.n_smem = sh.n_fill;
  };

  uint32_t lo_key = 0u;
  unsigned long long kept = (unsigned long long)V;
  if (use_k) {
    __syncthreads();
    if (warp == 0) choose_bucket(sh, false, 0.f);
    __syncthreads();
    for (int r = 1; r < 4; ++r) {
      if (tid == 0) sh.n_fill = 0;
      clear_hist();
      __syncthreads();
      round(false, 0u);
      if (warp == 0) choose_bucket(sh, false, 0.f);
      __syncthreads();
    }
    lo_key = sh.sel.prefix;
    kept = sh.sel.n_cand;
  }
  if (use_p) {
    __syncthreads();
    if (tid == 0) sh.sel = Select{0u, 0, 0ull, 0ull, 0ull, kept};
    for (int r = 0; r < 4; ++r) {
      if (tid == 0) sh.n_fill = 0;
      clear_hist();
      __syncthreads();
      round(true, lo_key);
      if (warp == 0) choose_bucket(sh, true, r == 0 ? p : 0.f);
      __syncthreads();
    }
    lo_key = sh.sel.prefix;
    kept = sh.sel.n_cand;
  }

  // ---- final pass over {z >= tau}: Gumbel-max and the kept set's mass ----
  Pick best{-INFINITY, 0x7fffffff};
  float best_z = 0.f;
  unsigned long long S = 0;
  for_each([&](float z, int id) {
    if (order_key(z) < lo_key) return;
    S += fixed_mass(z, M);
    const Pick nb = better(best, Pick{z + gumbel(seed, step, (uint32_t)b, (uint32_t)id), id});
    if (nb.i != best.i) best_z = z;
    best = nb;
  });
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const Pick other{__shfl_xor_sync(0xffffffffu, best.v, o), __shfl_xor_sync(0xffffffffu, best.i, o)};
    const float other_z = __shfl_xor_sync(0xffffffffu, best_z, o);
    S += __shfl_xor_sync(0xffffffffu, S, o);
    const Pick nb = better(best, other);
    if (nb.i != best.i) best_z = other_z;
    best = nb;
  }
  if (lane == 0) { sh.red_v[warp] = best.v; sh.red_i[warp] = best.i; sh.red_f[warp] = best_z; sh.red_m[warp] = S; }
  __syncthreads();
  if (tid == 0) {
    Pick bb{-INFINITY, 0x7fffffff};
    float bz = 0.f;
    unsigned long long tot = 0;
    for (int w = 0; w < kFilterThreads / 32; ++w) {
      const Pick nb = better(bb, Pick{sh.red_v[w], sh.red_i[w]});
      if (nb.i != bb.i) bz = sh.red_f[w];
      bb = nb;
      tot += sh.red_m[w];
    }
    const float lse = M + (float)(log((double)tot) - 40.0 * 0.69314718055994530942);
    out_ids[b] = bb.i;
    out_logprobs[b] = bz - lse;
    if (out_kept) out_kept[b] = (int32_t)kept;
  }
}

}  // namespace
}  // namespace prl

using namespace prl;

extern "C" size_t prl_sample_filter_workspace_bytes(int32_t B, int32_t V) {
  (void)B;
  (void)V;
  return 0;   // all per-row state lives in shared memory
}

extern "C" int prl_sample_filter_rows(const float* logits, int32_t B, int32_t V, const float* inv_temperature_rows,
                                      const uint8_t* greedy_rows, const int32_t* top_k_rows, const float* top_p_rows,
                                      uint64_t seed, uint32_t step, int32_t* out_ids, float* out_logprobs,
                                      int32_t* out_kept, void* workspace, size_t workspace_bytes, prl_stream_t st) {
  PRL_CHECK_ARG(logits && inv_temperature_rows && greedy_rows && top_k_rows && top_p_rows && out_ids && out_logprobs,
                "prl_sample_filter_rows: NULL argument");
  PRL_CHECK_ARG(B >= 1 && V >= 1, "prl_sample_filter_rows: bad shape (B %d, V %d)", B, V);
  PRL_CHECK_ARG(V <= kFilterMaxVocab, "prl_sample_filter_rows: vocabulary of %d exceeds %d", V, kFilterMaxVocab);
  PRL_CHECK_ARG(workspace_bytes >= prl_sample_filter_workspace_bytes(B, V) && (workspace || workspace_bytes == 0),
                "prl_sample_filter_rows: workspace too small");
  const int smem = kFilterCap * (int)(sizeof(float) + sizeof(int));
  static SmemAttr smem_attr = {};
  PRL_CUDA(ensure_smem(sample_filter_kernel, smem, smem_attr));
  PRL_CUDA(launch_pdl(sample_filter_kernel, dim3((unsigned)B), dim3(kFilterThreads), (size_t)smem, (cudaStream_t)st,
                      logits, (int)V, inv_temperature_rows, greedy_rows, top_k_rows, top_p_rows, seed, step, out_ids,
                      out_logprobs, out_kept));
  PRL_LAUNCH_CHECK();
  return PRL_OK;
}
