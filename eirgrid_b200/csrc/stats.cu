// stats.cu — per-batch update statistics accumulated on the device (sm_100a).
//
// The reference applies apply_contrast_learning / apply_deficit_contrast_learning (weights/learning.rs:131-373)
// one episode at a time under a write lock (core/multi_simulation.rs:494-508). For a batch sampled from one frozen
// snapshot and sharded over GPUs, the per-episode effect on the weight table is summarised here as a small integer
// table (DESIGN.md §update) that ranks sum with one NCCL allreduce:
//   header[0] episodes, header[1] episodes whose deterioration passed the contrast threshold, header[2] flagged episodes
//   per year: [0,61)    sum of ln(penalty_e)      over penalised occurrences of action k   (fixed point, 2^-24)
//             [61,122)  sum of ln(mild_penalty_e) over mis-positioned occurrences of k      (fixed point)
//             [122,183) occurrences of action k in current_run_actions
//             [183,198) occurrences of deficit key k in current_deficit_actions
// Integer sums make the result independent of the reduction order and of the number of GPUs.
#include "stats.cuh"
#include "update_rule.hpp"
#include <algorithm>

namespace {

__device__ __forceinline__ double default_score(const eg_result& r, double ln100, bool cost_only = false) {  // scoring.rs:5-44
  if (cost_only) return 2.0 - fmin(log(fmax(r.total_cost / egrule::kMaxCost, 1.0)) / ln100, 1.0);
  if (r.net_emissions > 0.0) return 1.0 - fmin(r.net_emissions / egrule::kMaxEmissions, 1.0);
  const double normalized_cost = fmax(r.total_cost / egrule::kMaxCost, 1.0);
  const double cost_score = 1.0 - fmin(log(normalized_cost) / ln100, 1.0);
  const double cost_weight = normalized_cost > 8.0 ? 0.8 : 0.5;
  return 1.0 + (cost_score * cost_weight + r.public_opinion * (1.0 - cost_weight));
}

__global__ void eg_stats_reset_kernel(double* best_score, unsigned long long* best_index) {
  *best_score = -1.0;
  *best_index = ~0ull;
}

// One episode per WARP: its ~40 recorded actions are dealt out to the lanes (a thread- or year-per-lane mapping runs at
// 1-3 active lanes because 2025 holds a third of an episode's actions), each lane folds its action into the block's
// shared accumulator. Grid-stride over the batch.
__global__ void __launch_bounds__(256) eg_stats_kernel(const EgStatsParams p) {
  __shared__ unsigned long long acc[EG_STATS_WORDS];
  __shared__ unsigned long long best_mask[EG_NY];                      // actions that occur in best(y) = best_actions ++ best_deficit
  __shared__ uint8_t best_cat[EG_BEST_CAPACITY + EG_TRAJ_CAPACITY];    // that concatenation by position, year after year
  __shared__ uint16_t best_len[EG_NY], best_start[EG_NY];
  for (int i = threadIdx.x; i < EG_STATS_WORDS; i += blockDim.x) acc[i] = 0ull;
  if (threadIdx.x < EG_NY) {
    const int y = threadIdx.x;
    const int nb = p.policy->n_best[y], nbd = p.policy->n_best_deficit[y];
    const int ob = p.policy->best_off[y], obd = p.policy->best_deficit_off[y];
    uint8_t* cat = best_cat + ob + obd;  // both offsets are prefix sums over the years before y
    unsigned long long m = 0ull;
    for (int b = 0; b < nb; b++) { const int a = p.policy->best[ob + b]; cat[b] = (uint8_t)a; m |= 1ull << a; }
    for (int b = 0; b < nbd; b++) { const int a = p.policy->best_deficit[obd + b]; cat[nb + b] = (uint8_t)a; m |= 1ull << a; }
    best_mask[y] = m;
    best_len[y] = (uint16_t)(nb + nbd);
    best_start[y] = (uint16_t)(ob + obd);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const uint32_t warps_total = gridDim.x * (blockDim.x >> 5);
  double warp_best = -1.0;
  for (uint32_t ep = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); ep < p.n; ep += warps_total) {
    const eg_result* rp = p.results + ep;
    eg_result r;  // every lane reads the same 40 bytes (one broadcast transaction)
    r.net_emissions = rp->net_emissions; r.public_opinion = rp->public_opinion; r.total_cost = rp->total_cost;
    const double score = default_score(r, p.ln100, p.consts.cost_only != 0);
    warp_best = fmax(warp_best, score);
    bool pass = false;
    long long log_pen = 0, log_mild = 0;
    if (p.consts.has_best) {
      const double det = p.consts.best_score > 0.0 ? (p.consts.best_score - score) / p.consts.best_score : 0.0;
      pass = det > p.consts.threshold || p.consts.force;
      if (pass) {
        if (det < 0.0) {
          // powf(negative, 0.3) is NaN and f64::max(NaN, MIN_WEIGHT) == MIN_WEIGHT (quirk Q9): collapse to the floor
          log_pen = log_mild = -(1ll << 40);
        } else {
          const double combined = pow(det, 0.3) * p.consts.stagnation;
          const double penalty = 1.0 / (1.0 + p.consts.alr * 1.5 * combined);
          const double mild = 1.0 / (1.0 + p.consts.alr * combined * 0.5);
          log_pen = llrint(log(penalty) * EG_STATS_FIXED_SCALE);
          log_mild = llrint(log(mild) * EG_STATS_FIXED_SCALE);
        }
      }
    }
    if (lane == 0) {
      atomicAdd(&acc[0], 1ull);
      if (pass) atomicAdd(&acc[1], 1ull);
      if (rp->flags) atomicAdd(&acc[2], 1ull);  // capacity overflow / no site: counted so that a driver can report it
    }
    // The episode's records: current_run_actions ++ current_deficit_actions of every year, ~40 items in all, most of them
    // in 2025. Lane y holds year y's counts; the items are numbered through all years (warp prefix sum) and dealt out 32 at
    // a time, each lane finding its item's year by binary search over the prefix sums.
    const eg_traj* t = p.trajs + ep;
    int nd = 0, nrun = 0;
    if (lane < EG_NY) { nd = t->n_deficit[lane]; nrun = nd + t->n_additional[lane]; }
    // first slot of each year's row in the record (rows are stored back to back); counts that run past the capacity
    // (never written by the episode kernels) are cut
    int row_end = nrun;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xFFFFFFFFu, row_end, o);
      if (lane >= o) row_end += v;
    }
    int row = row_end - nrun;
    if (row > EG_TRAJ_CAPACITY) row = EG_TRAJ_CAPACITY;
    if (row + nrun > EG_TRAJ_CAPACITY) { nrun = EG_TRAJ_CAPACITY - row; nd = min(nd, nrun); }
    const int cnt = nrun + nd;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
      if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    for (int base = 0; base < total; base += 32) {
      const int q = base + lane;
      int y = 0;  // number of years whose items all come before item q
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const int v = __shfl_sync(0xFFFFFFFFu, incl, y + step - 1);
        if (v <= q) y += step;
      }
      const int y_incl = __shfl_sync(0xFFFFFFFFu, incl, y), y_cnt = __shfl_sync(0xFFFFFFFFu, cnt, y);
      const int y_nrun = __shfl_sync(0xFFFFFFFFu, nrun, y), y_row = __shfl_sync(0xFFFFFFFFu, row, y);
      if (q >= total) continue;
      const int i = q - (y_incl - y_cnt);
      const int a = t->actions[y_row + (i < y_nrun ? i : i - y_nrun)];
      if (a >= EG_N_ACTIONS) continue;  // not an action code (records are produced by the episode kernels; defensive)
      unsigned long long* ys = acc + EG_STATS_HEADER + y * EG_STATS_YEAR_STRIDE;
      if (i < y_nrun) atomicAdd(&ys[2 * EG_N_ACTIONS + a], 1ull);
      else {
        const int k = egrule::deficit_key_of_action(a);
        if (k >= 0) atomicAdd(&ys[3 * EG_N_ACTIONS + k], 1ull);
      }
      if (!pass) continue;
      if (!((best_mask[y] >> a) & 1ull)) {
        atomicAdd(&ys[a], (unsigned long long)log_pen);
      } else if (i < (int)best_len[y]) {
        if (best_cat[best_start[y] + i] != a) atomicAdd(&ys[EG_N_ACTIONS + a], (unsigned long long)log_mild);
      }
    }
  }
  if (lane == 0 && warp_best >= 0.0) atomicMax((long long*)p.best_score, __double_as_longlong(warp_best));  // scores are >= 0: bit order == value order
  __syncthreads();
  for (int i = threadIdx.x; i < EG_STATS_WORDS; i += blockDim.x)
    if (acc[i]) atomicAdd((unsigned long long*)&p.stats[i], acc[i]);
}

__global__ void __launch_bounds__(256) eg_stats_argbest_kernel(const EgStatsParams p) {
  const uint32_t ep = blockIdx.x * blockDim.x + threadIdx.x;
  if (ep >= p.n) return;
  const double score = default_score(p.results[ep], p.ln100, p.consts.cost_only != 0);
  if (score == *p.best_score) atomicMin(p.best_index, (unsigned long long)ep);
}

__global__ void __launch_bounds__(320) eg_stats_pack_best_kernel(const eg_result* results, const eg_traj* trajs, uint32_t n, const double* best_score,
                                                                 const unsigned long long* best_index, unsigned long long first_global, uint32_t* record) {
  // 16 + 64 + 1088 bytes = 292 words, one per thread
  const unsigned long long raw = *best_index;
  const uint32_t idx = raw < n ? (uint32_t)raw : (n ? n - 1 : 0);
  const int w = threadIdx.x;
  constexpr int kRes = (int)sizeof(eg_result) / 4, kTraj = (int)sizeof(eg_traj) / 4;
  if (w < 2) record[w] = ((const uint32_t*)best_score)[w];
  else if (w < 4) { const unsigned long long g = first_global + idx; record[w] = (uint32_t)(g >> (32 * (w - 2))); }
  else if (w < 4 + kRes) record[w] = ((const uint32_t*)(results + idx))[w - 4];
  else if (w < 4 + kRes + kTraj) record[w] = ((const uint32_t*)(trajs + idx))[w - 4 - kRes];
}

// block b of rank r: r's buffer -> slot r of peer b's gather buffer (half `epoch & 1`), then flag r on peer b, then wait for
// flag b on r. The two halves alternate: a rank cannot start epoch e + 2 before every peer has started e + 1, i.e. has
// finished reading e (stream order on the peer), so a half is never overwritten while it is read.
__global__ void __launch_bounds__(256) eg_pack_exchange_kernel(const EgExchangeParams p) {
  constexpr int kRec = (int)(EG_BEST_RECORD_BYTES / 8), kWords = EG_STATS_WORDS + kRec;
  constexpr int kRes = (int)sizeof(eg_result) / 8;
  const uint32_t peer = blockIdx.x;
  const unsigned long long raw = *p.best_index;
  const uint32_t idx = raw < p.n ? (uint32_t)raw : (p.n ? p.n - 1 : 0);
  long long* dst = (long long*)p.peer_buf[peer] + ((size_t)(p.epoch & 1u) * p.world + p.rank) * kWords;
  const long long* res = (const long long*)(p.results + idx);
  const long long* trj = (const long long*)(p.trajs + idx);
  for (int i = threadIdx.x; i < kWords; i += blockDim.x) {
    long long v;
    if (i < EG_STATS_WORDS) v = p.stats[i];
    else {
      const int w = i - EG_STATS_WORDS;  // [score f64 | global id i64 | eg_result | eg_traj]
      v = w == 0 ? __double_as_longlong(*p.best_score) : w == 1 ? (long long)(p.first_global + idx) : w < 2 + kRes ? res[w - 2] : trj[w - 2 - kRes];
    }
    dst[i] = v;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t* remote = (uint32_t*)p.peer_flag[peer] + p.rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(remote), "r"(p.epoch) : "memory");
    const uint32_t* mine = (const uint32_t*)p.peer_flag[p.rank] + peer;
    const long long t0 = clock64();
    for (;;) {
      uint32_t v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if ((int32_t)(v - p.epoch) >= 0) break;
      if (clock64() - t0 > 4000000000ll) { *p.error = 1u; break; }  // ~2 s: a peer that never arrives must not hang the GPU
    }
  }
}

}  // namespace

cudaError_t eg_launch_pack_exchange(const EgExchangeParams& p, cudaStream_t stream) {
  static_assert(EG_BEST_RECORD_BYTES % 8 == 0 && sizeof(eg_result) % 8 == 0 && sizeof(eg_traj) % 8 == 0, "the record is copied in 64-bit words");
  if (p.world == 0 || p.world > EG_MAX_PEERS || p.rank >= p.world) return cudaErrorInvalidValue;
  eg_pack_exchange_kernel<<<p.world, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t eg_launch_pack_best(const eg_result* results, const eg_traj* trajs, uint32_t n, const double* best_score,
                                const unsigned long long* best_index, unsigned long long first_global, void* record, cudaStream_t stream) {
  static_assert(sizeof(eg_result) % 4 == 0 && sizeof(eg_traj) % 4 == 0, "record is copied in 32-bit words");
  eg_stats_pack_best_kernel<<<1, 320, 0, stream>>>(results, trajs, n, best_score, best_index, first_global, (uint32_t*)record);
  return cudaGetLastError();
}

cudaError_t eg_launch_stats(const EgStatsParams& p, cudaStream_t stream) {
  eg_stats_reset_kernel<<<1, 1, 0, stream>>>(p.best_score, p.best_index);
  if (p.n == 0) return cudaGetLastError();
  const uint32_t blocks = (p.n + 255) / 256;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const uint32_t stat_blocks = std::min<uint32_t>((uint32_t)sms * 4u, (p.n + 7) / 8);  // 8 warps (episodes) per block, grid-stride
  eg_stats_kernel<<<stat_blocks, 256, 0, stream>>>(p);
  eg_stats_argbest_kernel<<<blocks, 256, 0, stream>>>(p);
  return cudaGetLastError();
}
