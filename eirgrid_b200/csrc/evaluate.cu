// evaluate.cu — policy evaluation: rollout outputs reduced into an eg_eval_stats record on the device (sm_100a), and the host
// merge of two records.
//
// Two kernels per chunk of at most EG_EVAL_CHUNK episodes:
//   block pass  block b takes the contiguous slice [b * EG_EVAL_SLICE, (b + 1) * EG_EVAL_SLICE) of the chunk. Integer counters
//               (flags, score histogram, per-year counts, action counts) go through shared-memory atomics and then one global
//               atomic per nonzero word into the record: sums of integers, independent of the order. Each moment entry (9
//               final metrics, 26 x 18 yearly fields) is folded by one thread over the slice in episode order (Welford).
//   fold pass   one thread per moment entry merges the block partials into the record in block order (Chan et al.).
// The partition depends on n only, never on the SM count or the launch timing, so the record is the same bytes on every run.
#include "evaluate.cuh"
#include <cstring>
#include "common.hpp"
#include "traj_rows.hpp"

namespace {

// word of a counter in the counter part of the record (n_flagged .. end)
#define EG_EVAL_WORD(field) ((int)((offsetof(eg_eval_stats, field) - offsetof(eg_eval_stats, n_flagged)) / sizeof(uint64_t)))

// where moment entry e lies in an episode's records: byte offset, record stride, and the type (0 f64, 1 u32, 2 u16)
struct EntrySource {
  size_t offset, stride;
  int kind;
};

__device__ __forceinline__ EntrySource entry_source(int e) {
  if (e < 5) return {offsetof(eg_result, score) + sizeof(double) * e, sizeof(eg_result), 0};  // the five f64 fields in order
  if (e < 7) return {offsetof(eg_result, n_generators) + sizeof(uint32_t) * (e - 5), sizeof(eg_result), 1};
  if (e < EG_EVAL_N_FINAL) return {offsetof(eg_result, n_deficit_actions) + sizeof(uint16_t) * (e - 7), sizeof(eg_result), 2};
  const int y = (e - EG_EVAL_N_FINAL) / EG_EVAL_N_YEAR_FIELDS, f = (e - EG_EVAL_N_FINAL) % EG_EVAL_N_YEAR_FIELDS;
  const size_t year = sizeof(eg_year_metrics) * y;
  if (f < 2) return {year + offsetof(eg_year_metrics, total_population) + sizeof(uint32_t) * f, sizeof(eg_yearly), 1};
  return {year + offsetof(eg_year_metrics, total_power_usage) + sizeof(double) * (f - 2), sizeof(eg_yearly), 0};
}

__device__ __forceinline__ double load_value(const unsigned char* p, int kind) {
  if (kind == 0) return __ldg((const double*)p);
  if (kind == 1) return (double)__ldg((const unsigned int*)p);
  return (double)__ldg((const unsigned short*)p);
}

__global__ void __launch_bounds__(EG_EVAL_SLICE) eg_eval_block_kernel(const EgEvalParams p) {
  constexpr int kFlagged = EG_EVAL_WORD(n_flagged), kFlags = EG_EVAL_WORD(flag_counts), kHist = EG_EVAL_WORD(score_hist),
                kOut = EG_EVAL_WORD(score_out_of_range), kNetZero = EG_EVAL_WORD(net_zero_or_below),
                kDeficit = EG_EVAL_WORD(in_deficit), kFirst = EG_EVAL_WORD(first_net_zero_year),
                kAdd = EG_EVAL_WORD(additional_actions), kDefAct = EG_EVAL_WORD(deficit_actions);
  __shared__ unsigned int cnt[EG_EVAL_COUNTER_WORDS];  // a block counts at most 256 x 984 actions: 32 bits suffice
  for (int i = threadIdx.x; i < EG_EVAL_COUNTER_WORDS; i += blockDim.x) cnt[i] = 0u;
  __syncthreads();
  const uint32_t lo = blockIdx.x * EG_EVAL_SLICE, hi = min(p.n, lo + EG_EVAL_SLICE);
  const int lane = threadIdx.x & 31;
  // counters of the episode's result and yearly records: one thread per episode
  if (lo + threadIdx.x < hi) {
    const uint32_t ep = lo + threadIdx.x;
    const eg_result& r = p.results[ep];
    if (r.flags) {
      atomicAdd(&cnt[kFlagged], 1u);
      for (int b = 0; b < EG_EVAL_N_FLAGS; b++)
        if ((r.flags >> b) & 1u) atomicAdd(&cnt[kFlags + b], 1u);
    }
    const double s = r.score;  // s * 1024 is exact; truncation is floor for s >= 0
    if (s >= 0.0 && s <= 2.0) atomicAdd(&cnt[kHist + min((int)(s * 1024.0), EG_EVAL_SCORE_BINS - 1)], 1u);
    else atomicAdd(&cnt[kOut], 1u);
    if (p.yearly) {
      int first = EG_NY;
      for (int y = EG_NY - 1; y >= 0; y--) {
        const eg_year_metrics& ym = p.yearly[ep].y[y];
        if (ym.net_co2_emissions <= 0.0) { atomicAdd(&cnt[kNetZero + y], 1u); first = y; }
        if (ym.power_balance < 0.0) atomicAdd(&cnt[kDeficit + y], 1u);
      }
      atomicAdd(&cnt[kFirst + first], 1u);
    }
  }
  // counters of the action records: one warp per episode
  for (uint32_t ep = lo + (threadIdx.x >> 5); ep < hi; ep += EG_EVAL_SLICE / 32) {
    // the action records: row slots [0, nd) are the deficit actions, [nd, nrun) the additional ones; the items past the row
    // repeat the deficit actions and are the ones counted as such
    eg_warp_traj_items(p.traj + ep, lane, [&](int y, int i, int nrun, int nd, int a) {
      if (a >= EG_N_ACTIONS) return;
      if (i >= nrun) atomicAdd(&cnt[kDefAct + y * EG_N_ACTIONS + a], 1u);
      else if (i >= nd) atomicAdd(&cnt[kAdd + y * EG_N_ACTIONS + a], 1u);
    });
  }
  // moments: one thread per entry, the slice in episode order (Welford)
  const uint32_t count = hi - lo;
  const int n_entries = p.yearly ? egeval::kMoments : EG_EVAL_N_FINAL;
  for (int e = threadIdx.x; e < n_entries; e += EG_EVAL_SLICE) {
    const EntrySource src = entry_source(e);
    const unsigned char* base =
        (e < EG_EVAL_N_FINAL ? (const unsigned char*)(p.results + lo) : (const unsigned char*)(p.yearly + lo)) + src.offset;
    eg_moments m{0.0, 0.0, 0.0, 0.0};
    uint32_t best = 0, worst = 0;
    for (uint32_t k0 = 0; k0 < count; k0 += 8) {
      double x[8];
#pragma unroll
      for (int j = 0; j < 8; j++) x[j] = k0 + j < count ? load_value(base + (size_t)(k0 + j) * src.stride, src.kind) : 0.0;
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const uint32_t k = k0 + j;
        if (k >= count) break;
        if (k == 0) {
          m.mean = x[j]; m.m2 = 0.0; m.min = x[j]; m.max = x[j];
          continue;
        }
        const double d = x[j] - m.mean;
        m.mean = m.mean + d / (double)(k + 1);
        m.m2 = m.m2 + d * (x[j] - m.mean);
        if (egeval::below(m.min, x[j])) { m.min = x[j]; worst = k; }
        if (egeval::above(m.max, x[j])) { m.max = x[j]; best = k; }
      }
    }
    EgEvalPartial& out = p.partials[blockIdx.x];
    out.m[e] = m;
    if (e == 0) {
      out.best = p.first_global + lo + best;
      out.worst = p.first_global + lo + worst;
    }
  }
  __syncthreads();
  unsigned long long* acc = (unsigned long long*)egeval::counters(p.acc);
  for (int i = threadIdx.x; i < EG_EVAL_COUNTER_WORDS; i += blockDim.x)
    if (cnt[i]) atomicAdd(&acc[i], (unsigned long long)cnt[i]);
}

// one block: thread e merges the partials of moment entry e into the record in block order
__global__ void __launch_bounds__(512) eg_eval_fold_kernel(const EgEvalParams p) {
  static_assert(egeval::kMoments <= 512, "one thread per moment entry");
  eg_eval_stats* acc = p.acc;
  const uint64_t n0 = acc->n_episodes;
  const bool yearly = p.yearly != nullptr && (n0 == 0 || acc->has_yearly);
  const uint32_t blocks = (p.n + EG_EVAL_SLICE - 1) / EG_EVAL_SLICE;
  const int e = threadIdx.x;
  if (e < (yearly ? egeval::kMoments : EG_EVAL_N_FINAL)) {
    eg_moments m = egeval::moments(acc)[e];
    uint64_t best = acc->best_episode, worst = acc->worst_episode;
    uint64_t na = n0;
    for (uint32_t b0 = 0; b0 < blocks; b0 += 8) {
      eg_moments mb[8];  // eight partials loaded ahead of their merges, so that the loads overlap
#pragma unroll
      for (int j = 0; j < 8; j++)
        if (b0 + j < blocks) mb[j] = p.partials[b0 + j].m[e];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const uint32_t b = b0 + j;
        if (b >= blocks) break;
        const uint64_t nb = min((uint32_t)EG_EVAL_SLICE, p.n - b * EG_EVAL_SLICE);
        if (e == 0) egeval::merge_extreme_ids(best, worst, m, na, p.partials[b].best, p.partials[b].worst, mb[j], nb);
        egeval::merge_moments(m, na, mb[j], nb);
        na += nb;
      }
    }
    egeval::moments(acc)[e] = m;
    if (e == 0) { acc->best_episode = best; acc->worst_episode = worst; }
  }
  __syncthreads();  // every thread has read n_episodes and has_yearly
  if (threadIdx.x == 0) {
    acc->n_episodes = n0 + p.n;
    acc->has_yearly = (n0 == 0 ? p.yearly != nullptr : acc->has_yearly && p.yearly != nullptr) ? 1u : 0u;
  }
}

}  // namespace

cudaError_t eg_launch_eval(const EgEvalParams& p, cudaStream_t stream) {
  if (p.n == 0) return cudaSuccess;
  if (p.n > EG_EVAL_CHUNK) return cudaErrorInvalidValue;
  eg_eval_block_kernel<<<(p.n + EG_EVAL_SLICE - 1) / EG_EVAL_SLICE, EG_EVAL_SLICE, 0, stream>>>(p);
  eg_eval_fold_kernel<<<1, 512, 0, stream>>>(p);
  return cudaGetLastError();
}

extern "C" int eg_eval_stats_merge(eg_eval_stats* dst, const eg_eval_stats* src) {
  if (!dst || !src) return eg_fail(EG_ERR_INVALID, "eg_eval_stats_merge: NULL argument");
  if (src->n_episodes == 0) return EG_OK;
  if (dst->n_episodes == 0) {
    std::memcpy(dst, src, sizeof(eg_eval_stats));
    return EG_OK;
  }
  if ((dst->has_yearly != 0) != (src->has_yearly != 0))
    return eg_fail(EG_ERR_INVALID, "eg_eval_stats_merge: only one of the records has the per-year part");
  const uint64_t na = dst->n_episodes, nb = src->n_episodes;
  uint64_t best = dst->best_episode, worst = dst->worst_episode;
  egeval::merge_extreme_ids(best, worst, dst->final_metrics[0], na, src->best_episode, src->worst_episode, src->final_metrics[0], nb);
  dst->best_episode = best;
  dst->worst_episode = worst;
  const int n_entries = dst->has_yearly ? egeval::kMoments : EG_EVAL_N_FINAL;
  for (int e = 0; e < n_entries; e++) egeval::merge_moments(egeval::moments(dst)[e], na, egeval::moments(src)[e], nb);
  for (int i = 0; i < EG_EVAL_COUNTER_WORDS; i++) egeval::counters(dst)[i] += egeval::counters(src)[i];
  dst->n_episodes = na + nb;
  return EG_OK;
}
