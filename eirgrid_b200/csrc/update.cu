// update.cu — the reference's per-episode weight update, applied in episode order ON THE DEVICE (sm_100a).
//
// Reference: the write-lock section of the batch driver, core/multi_simulation.rs:494-508, for every episode in turn:
//   transfer_recorded_actions_from (weights/strategy.rs:313-342) -> apply_contrast_learning (weights/learning.rs:131-283)
//   -> update_best_strategy (strategy.rs:19-258) -> apply_deficit_contrast_learning (learning.rs:285-373).
// The host form of the same rule is eg_update (weights.cpp); this file ends with the same table, bit for bit, because the
// scalar part of the rule comes from the shared update_rule.hpp / eg_math.hpp and every table entry receives the same
// multiplications in the same order.
//
// How a strictly sequential rule is spread over a GPU:
//   * What an episode's update does depends on the episodes before it only through (a) which strategy is the best so
//     far, its score and the stagnation counter — functions of the SCORES alone (a running strict maximum) — and (b) the
//     table entries themselves, where entry (year, action) only ever sees its own history.
//   * So one pass is: scores (parallel) -> prefix maximum with the index of the episode that holds it (one block scan)
//     -> per-episode thresholds and factors (parallel, exp/pow here) -> best-strategy lists of the improving episodes
//     (parallel) -> per (episode, year) the NUMBER of penalty multiplications each entry receives, from comparing the
//     episode's record with the strategy that was best when its turn came (parallel, one warp per episode)
//     -> the table walk: one block per year, one thread per entry, episodes in order. The walk is the only serial part
//     and touches nothing but its own stream of 64-byte control records and 80-byte count rows, staged through shared
//     memory by bulk asynchronous copies (cp.async.bulk + mbarrier, three stages), plus one weight in a register. The
//     factors of the randomisation branch (one Philox draw per table entry and episode) are produced by a parallel kernel
//     beforehand and stream in the same way.
#include "update.cuh"
#include "traj_rows.hpp"
#include "update_rule.hpp"
#include <cstddef>

namespace {

constexpr int kWalkThreads = 96;   // 61 action entries (threads 0-60) and 15 deficit entries (threads 64-78) of one year
constexpr int kWalkTile = 64;      // episodes per stage
constexpr int kWalkStages = 3;
constexpr int kCtlBytes = (int)sizeof(EgUpdCtl);
static_assert(sizeof(EgUpdCtl) == 64, "control records are copied in bulk: 16-byte multiples");
static_assert(EG_UPD_ROW % 16 == 0 && EG_UPD_ROW >= EG_N_ACTIONS + EG_N_DEFICIT_KEYS, "count rows are copied in bulk");
static_assert(sizeof(EgUpdSlot) % 8 == 0, "slots are copied in 64-bit words");

struct Best2 {   // running strict maximum and the first episode that holds it
  double v;
  int i;
};
__device__ __forceinline__ Best2 later_if_greater(Best2 earlier, Best2 later) { return (later.v > earlier.v) ? later : earlier; }
__device__ __forceinline__ Best2 shfl_up_best(Best2 b, int o) {
  Best2 r;
  r.v = __shfl_up_sync(0xFFFFFFFFu, b.v, o);
  r.i = __shfl_up_sync(0xFFFFFFFFu, b.i, o);
  return r;
}
__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xFFF0000000000000ll); }

// ---- 1. scores ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) upd_score_kernel(const eg_result* results, uint32_t n, double* score, EgUpdState* st) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const eg_result* r = results + e;
  const double m[4] = {r->net_emissions, r->public_opinion, r->total_cost, r->power_reliability};
  score[e] = egrule::score(m, st->cost_only != 0);
  if (r->flags) atomicAdd(&st->n_flagged, 1u);
}

// ---- 2. running best: one block, every thread a contiguous piece of the pass ------------------------------------------
__global__ void __launch_bounds__(1024) upd_scan_kernel(const eg_result* results, uint32_t n, uint32_t base, EgUpdBuffers b) {
  __shared__ Best2 warp_best[32];
  __shared__ int warp_count[32];
  __shared__ Best2 pass_best;
  EgUpdState* st = b.state;
  const uint32_t has_best0 = st->has_best, iwi0 = st->iwi, it0 = st->iteration_count, improvements0 = st->n_improvements;
  const double best0 = st->best_score;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint32_t per = (n + 1023u) / 1024u;
  const uint32_t lo = min((uint32_t)t * per, n), hi = min(lo + per, n);
  Best2 mine = {neg_inf(), -1};
  for (uint32_t e = lo; e < hi; e++) mine = later_if_greater(mine, Best2{b.score[e], (int)e});
  Best2 inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const Best2 other = shfl_up_best(inc, o);
    if (lane >= o) inc = later_if_greater(other, inc);
  }
  if (lane == 31) warp_best[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    Best2 w = warp_best[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const Best2 other = shfl_up_best(w, o);
      if (lane >= o) w = later_if_greater(other, w);
    }
    warp_best[lane] = w;  // inclusive over warps
    if (lane == 31) pass_best = w;
  }
  __syncthreads();
  Best2 run = has_best0 ? Best2{best0, -1} : Best2{neg_inf(), -1};
  if (warp > 0) run = later_if_greater(run, warp_best[warp - 1]);
  const Best2 before_me = shfl_up_best(inc, 1);
  if (lane > 0) run = later_if_greater(run, before_me);
  int improved_here = 0;
  for (uint32_t e = lo; e < hi; e++) {
    const double s = b.score[e];
    EgUpdPre p;
    p.best_before = run.v;
    p.improver = run.i;
    p.iwi_before = run.i < 0 ? iwi0 + e : e - (uint32_t)run.i - 1u;
    p.improved = s > run.v ? 1u : 0u;  // update_best_strategy: strictly greater, or no best strategy yet (run.v = -inf)
    p.pad = 0;
    b.pre[e] = p;
    if (p.improved) { run = Best2{s, (int)e}; improved_here++; }
  }
  // ordered list of the improving episodes (improvement_history): exclusive scan of the counts
  int cinc = improved_here;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int other = __shfl_up_sync(0xFFFFFFFFu, cinc, o);
    if (lane >= o) cinc += other;
  }
  if (lane == 31) warp_count[warp] = cinc;
  __syncthreads();
  if (warp == 0) {
    int w = warp_count[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int other = __shfl_up_sync(0xFFFFFFFFu, w, o);
      if (lane >= o) w += other;
    }
    warp_count[lane] = w;
  }
  __syncthreads();
  uint32_t slot = improvements0 + (uint32_t)(cinc - improved_here) + (warp > 0 ? (uint32_t)warp_count[warp - 1] : 0u);
  if (improved_here)
    for (uint32_t e = lo; e < hi; e++)
      if (b.pre[e].improved) {
        if (slot < b.improvements_capacity) {
          const eg_result* r = results + e;
          EgUpdImprovement rec;
          rec.episode = (long long)base + e;
          rec.score = b.score[e];
          rec.metrics[0] = r->net_emissions; rec.metrics[1] = r->public_opinion; rec.metrics[2] = r->total_cost; rec.metrics[3] = r->power_reliability;
          b.improvements[slot] = rec;
        }
        slot++;
      }
  if (t == 1023) {  // `run` of the last thread is the state after the whole pass
    st->pass_has_best = has_best0; st->pass_iwi = iwi0; st->pass_iteration_count = it0;
    st->pass_any_random = 0u;
    st->pass_last_improver = run.i;
    if (run.i >= 0) {
      const eg_result* r = results + run.i;
      st->has_best = 1u;
      st->best_score = run.v;
      st->best_metrics[0] = r->net_emissions; st->best_metrics[1] = r->public_opinion; st->best_metrics[2] = r->total_cost; st->best_metrics[3] = r->power_reliability;
      st->iwi = n - 1u - (uint32_t)run.i;
    } else {
      st->iwi = iwi0 + n;
    }
    st->iteration_count = it0 + n;
    st->n_improvements = improvements0 + (uint32_t)warp_count[31];
    if (n && (st->batch_best_index < 0 || pass_best.v > st->batch_best_score)) {
      st->batch_best_score = pass_best.v;
      st->batch_best_index = (long long)base + pass_best.i;
    }
  }
}

// ---- 3. thresholds and factors of every episode -----------------------------------------------------------------------
__global__ void __launch_bounds__(128) upd_ctl_kernel(uint32_t n, EgUpdBuffers b) {
  const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  bool applied = false;
  if (e < n) {
    const EgUpdState* st = b.state;
    const EgUpdPre p = b.pre[e];
    const double lr = st->learning_rate;
    EgUpdCtl c;
    c.boost = c.penalty = c.mild = c.d_boost = c.d_penalty = 1.0;
    c.flags = p.improved ? EG_UPD_IMPROVED : 0u;
    c.iteration = st->pass_iteration_count + e;
    c.pad[0] = c.pad[1] = c.pad[2] = c.pad[3] = 0u;
    if (st->pass_has_best || p.improver >= 0) {  // apply_contrast_learning returns at once without a best strategy
      const egrule::Contrast k = egrule::contrast(p.best_before, b.score[e], p.iwi_before, lr);
      if (k.applied) {
        applied = true;
        c.flags |= EG_UPD_APPLIED | (k.randomise ? EG_UPD_RANDOMISE : 0u);
        c.boost = k.boost; c.penalty = k.penalty; c.mild = k.mild;
      }
    }
    const uint32_t iwi_after = p.improved ? 0u : p.iwi_before + 1u;
    const egrule::Contrast d = egrule::deficit_contrast(iwi_after, lr);
    if (d.applied) {
      c.flags |= EG_UPD_D_APPLIED | (d.randomise ? EG_UPD_D_RANDOMISE : 0u);
      c.d_boost = d.boost; c.d_penalty = d.penalty;
    }
    auto saturates = [](double boost) { return boost >= 1.0 && egrule::kMinWeight * boost >= egrule::kMaxWeight; };
    auto kills = [](double p) { return p != p || egrule::kMaxWeight * p <= egrule::kMinWeight; };
    if (saturates(c.boost)) c.flags |= EG_UPD_BOOST_SAT;
    if (kills(c.penalty)) c.flags |= EG_UPD_PEN_KILL;
    if (kills(c.mild)) c.flags |= EG_UPD_MILD_KILL;
    if (saturates(c.d_boost)) c.flags |= EG_UPD_D_BOOST_SAT;
    if (kills(c.d_penalty)) c.flags |= EG_UPD_D_PEN_KILL;
    if (c.boost >= 1.0 && !(c.penalty > 1.0) && !(c.mild > 1.0)) c.flags |= EG_UPD_PROPER;
    if (c.d_boost >= 1.0 && !(c.d_penalty > 1.0)) c.flags |= EG_UPD_D_PROPER;
    b.ctl[e] = c;
    if (c.flags & (EG_UPD_RANDOMISE | EG_UPD_D_RANDOMISE)) b.state->pass_any_random = 1u;  // same value from every writer
  }
  const unsigned m = __ballot_sync(0xFFFFFFFFu, applied);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(&b.state->n_applied, (uint32_t)__popc(m));
}

// ---- 4. best-strategy lists of the improving episodes (one warp per episode, lane = year) ------------------------------
__global__ void __launch_bounds__(256) upd_expand_kernel(const eg_traj* trajs, uint32_t n, uint32_t replay, EgUpdBuffers b) {
  const uint32_t e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (e >= n || !b.pre[e].improved) return;
  const eg_traj* t = trajs + e;
  EgUpdSlot* s = b.slots + e + 1;
  const EgTrajRow r = eg_warp_traj_row(t, lane);
  const uint8_t* a = t->actions + r.row;
  int len_run = 0, len_def = 0;
  unsigned long long mall = 0ull, mdef = 0ull;
  eg_for_each_run(a, r.nd, r.na, replay != 0, [&](int c) { len_run++; mall |= 1ull << c; });
  eg_for_each_deficit(a, r.nd, replay != 0, [&](int c) { len_def++; mdef |= 1ull << c; });
  int end = len_run + len_def;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xFFFFFFFFu, end, o);
    if (lane >= o) end += v;
  }
  if (lane >= EG_NY) return;
  const int off = end - (len_run + len_def);
  s->len_run[lane] = (uint16_t)len_run;
  s->len_def[lane] = (uint16_t)len_def;
  s->off[lane] = (uint32_t)off;
  s->mask_all[lane] = mall | mdef;
  s->mask_def[lane] = mdef;
  uint8_t* out = s->cat + off;
  int i = 0;
  eg_for_each_run(a, r.nd, r.na, replay != 0, [&](int c) { out[i++] = (uint8_t)c; });
  eg_for_each_deficit(a, r.nd, replay != 0, [&](int c) { out[i++] = (uint8_t)c; });
}

// Number of penalty / mild-penalty multiplications entry `key` of year `y` receives from one episode (learning.rs:228-262),
// and of deficit entry `dkey` (learning.rs:340-352): the slow, exact form used when a count does not fit a byte.
__device__ int count_regular(const uint8_t* a, int nd, int na, bool replay, const EgUpdSlot* s, int y, int key) {
  const uint8_t* B = s->cat + s->off[y];
  const int LB = s->len_run[y] + s->len_def[y];
  const bool in_best = (s->mask_all[y] >> key) & 1ull;
  int i = 0, cnt = 0;
  auto visit = [&](int c) {
    if (c == key && (!in_best || (i < LB && B[i] != c))) cnt++;
    i++;
  };
  eg_for_each_run(a, nd, na, replay, visit);
  eg_for_each_deficit(a, nd, replay, visit);
  return cnt;
}
__device__ int count_deficit(const uint8_t* a, int nd, bool replay, const EgUpdSlot* s, int y, int dkey) {
  const unsigned long long mdef = s->mask_def[y];
  int cnt = 0;
  eg_for_each_deficit(a, nd, replay, [&](int c) {
    if (!((mdef >> c) & 1ull) && egrule::deficit_key_of_action(c) == dkey) cnt++;
  });
  return cnt;
}

// ---- 5. multiplication counts per (episode, year, entry): one warp per episode, lane = year ---------------------------
constexpr int kPrepWarps = 8;
__global__ void __launch_bounds__(kPrepWarps * 32) upd_prep_kernel(const eg_traj* trajs, uint32_t n, uint32_t replay, EgUpdBuffers b) {
  __shared__ __align__(16) uint8_t rows[kPrepWarps][32][EG_UPD_ROW];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t e = blockIdx.x * kPrepWarps + w;
  if (e >= n) return;
  const uint32_t flags = b.ctl[e].flags;
  const eg_traj* t = trajs + e;
  const EgTrajRow yr = eg_warp_traj_row(t, lane);
  if (lane >= EG_NY) return;
  uint8_t* r = rows[w][lane];
  uint4* r4 = (uint4*)r;
#pragma unroll
  for (int q = 0; q < EG_UPD_ROW / 16; q++) r4[q] = make_uint4(0u, 0u, 0u, 0u);
  const uint8_t* a = t->actions + yr.row;
  const EgUpdSlot* s = b.slots + (b.pre[e].improver + 1);
  const bool rp = replay != 0;
  auto bump = [&](int idx) {
    const int v = r[idx];
    if (v < 255) r[idx] = (uint8_t)(v + 1);  // 255 = "count it again from the record" (the walk does)
  };
  if (flags & EG_UPD_APPLIED) {
    const uint8_t* B = s->cat + s->off[lane];
    const int LB = s->len_run[lane] + s->len_def[lane];
    const unsigned long long mall = s->mask_all[lane];
    int i = 0;
    auto visit = [&](int c) {
      if (!((mall >> c) & 1ull)) bump(c);                 // not part of the best strategy of this year: penalty
      else if (i < LB && B[i] != c) bump(c);              // part of it, at another position: mild penalty
      i++;
    };
    eg_for_each_run(a, yr.nd, yr.na, rp, visit);
    eg_for_each_deficit(a, yr.nd, rp, visit);
  }
  if (flags & EG_UPD_D_APPLIED) {
    const unsigned long long mdef = s->mask_def[lane];
    eg_for_each_deficit(a, yr.nd, rp, [&](int c) {
      if (!((mdef >> c) & 1ull)) {
        const int k = egrule::deficit_key_of_action(c);
        if (k >= 0) bump(EG_N_ACTIONS + k);
      }
    });
  }
  uint4* out = (uint4*)(b.counts + ((size_t)lane * EG_UPD_CHUNK + e) * EG_UPD_ROW);
#pragma unroll
  for (int q = 0; q < EG_UPD_ROW / 16; q++) out[q] = r4[q];
}

// ---- bulk asynchronous copies (TMA engine, 1-D form) and their mbarriers ---------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}

// ---- 6a. factors of the randomisation branch (learning.rs:267-280, 358-370), off the serial path ----------------------
// One thread per (episode, year, table entry): f = 1 + 0.25 (2u - 1) with u the entry's draw of the episode's stream.
// Only episodes whose flags ask for it are written; the walk never reads the others.
__global__ void __launch_bounds__(256) upd_random_kernel(uint32_t n, uint32_t key_lo, uint32_t key_hi, EgUpdBuffers b) {
  constexpr uint32_t kPerEpisode = EG_NY * EG_UPD_ENTRIES;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t e = t / kPerEpisode, r = t - e * kPerEpisode;
  if (e >= n) return;
  const uint32_t flags = b.ctl[e].flags;
  if (!(flags & (EG_UPD_RANDOMISE | EG_UPD_D_RANDOMISE))) return;
  const uint32_t y = r / EG_UPD_ENTRIES, k = r - y * EG_UPD_ENTRIES;
  uint32_t draw;
  if (k < EG_N_ACTIONS) {
    if (!(flags & EG_UPD_RANDOMISE)) return;
    draw = y * EG_N_ACTIONS + k;
  } else {
    if (!(flags & EG_UPD_D_RANDOMISE)) return;
    // the deficit table draws after the main table's 26 x 61 draws when both were randomised in this episode
    draw = ((flags & EG_UPD_RANDOMISE) ? (uint32_t)egrule::kContrastDraws : 0u) + y * EG_N_DEFICIT_KEYS + (k - EG_N_ACTIONS);
  }
  const double u = egrule::update_uniform(key_lo, key_hi, b.ctl[e].iteration, draw);
  b.factors[((size_t)y * EG_UPD_CHUNK + e) * EG_UPD_ENTRIES + k] = egrule::random_factor(u);
}

// ---- 6b. the table walk: block = year, thread = table entry, episodes in order -----------------------------------------
// A lone warp per scheduler issues one dependent instruction every ~6 cycles, so what counts here is the number of
// instructions per episode and that nothing but the entry's own value is waited for (walk_tile below).
struct WalkSmem {
  unsigned char ctl[kWalkStages][kWalkTile * kCtlBytes];
  unsigned char cnt[kWalkStages][kWalkTile * EG_UPD_ROW];
  double factors[kWalkStages][kWalkTile * EG_UPD_ENTRIES];  // only staged when the pass randomises at all
  unsigned long long full[kWalkStages];
};
static_assert(offsetof(WalkSmem, cnt) % 16 == 0 && offsetof(WalkSmem, factors) % 16 == 0 && offsetof(WalkSmem, full) % 8 == 0,
              "bulk copies need 16-byte aligned destinations");

// rare paths of the walk, kept out of line so that the episode loop stays short
template <bool DEFICIT>
__device__ __noinline__ int walk_recount(const eg_traj* t, int y, int key, bool rp, const EgUpdSlot* cur) {
  EgTrajRow r{};
  for (int yy = 0; yy <= y; yy++) r = eg_traj_next_row(*t, yy, r);
  const uint8_t* a = t->actions + r.row;
  return DEFICIT ? count_deficit(a, r.nd, rp, cur, y, key) : count_regular(a, r.nd, r.na, rp, cur, y, key);
}
template <bool DEFICIT>
__device__ __noinline__ int walk_occurrences(const EgUpdSlot* s, int y, int key) {
  int c = 0;
  if (!DEFICIT) {
    const uint8_t* B = s->cat + s->off[y];
    const int LB = s->len_run[y] + s->len_def[y];
    for (int i = 0; i < LB; i++) c += (B[i] == key);
  } else {
    const uint8_t* B = s->cat + s->off[y] + s->len_run[y];
    const int LB = s->len_def[y];
    for (int i = 0; i < LB; i++) c += (egrule::deficit_key_of_action(B[i]) == key);
  }
  return c;
}
__device__ __noinline__ double walk_boost(double w, double boost, int occ) {  // every occurrence in the best strategy (learning.rs:222-226)
  for (int q = 0; q < occ; q++) {
    if (w == egrule::kMaxWeight && boost >= 1.0) break;  // MAX_WEIGHT is a fixed point of the step
    w = egrule::min_std(w * boost, egrule::kMaxWeight);
  }
  return w;
}
__device__ __noinline__ double walk_penalty(double w, double pen, int m) {  // m penalty multiplications (learning.rs:228-262)
  for (int q = 0; q < m; q++) {
    if (w == egrule::kMinWeight && !(pen > 1.0)) break;  // MIN_WEIGHT is a fixed point (also for a NaN factor, quirk Q9)
    w = egrule::max_nan(w * pen, egrule::kMinWeight);
  }
  return w;
}

// One tile of up to 64 episodes for one table entry. The flags of the tile's episodes are first turned into bit masks that
// are the same in every thread of the warp (so the branches on them are uniform); the episodes are then visited in groups
// of eight whose operands — count byte, random factor, boost / penalty / mild penalty — are all fetched from shared
// memory BEFORE the group's multiplications start: the entry's value is the only dependency that runs through the loop.
template <bool DEFICIT>
__device__ __forceinline__ void walk_tile(const EgUpdCtl* ctl, const unsigned char* rows, const double* fac, uint32_t cnt, uint32_t first,
                                          int y, int key, bool live, bool rp, bool any_random, const eg_traj* trajs,
                                          const EgUpdBuffers& b, double& w, int& occ, const EgUpdSlot*& cur) {
  const int lane = threadIdx.x & 31;
  constexpr uint32_t kApplied = DEFICIT ? EG_UPD_D_APPLIED : EG_UPD_APPLIED;
  constexpr uint32_t kRandom = DEFICIT ? EG_UPD_D_RANDOMISE : EG_UPD_RANDOMISE;
  constexpr int kRowOffset = DEFICIT ? EG_N_ACTIONS : 0;
  constexpr int kGroup = 8;
  const unsigned char* my_rows = rows + kRowOffset + key;
  const double* my_fac = fac + kRowOffset + key;
#pragma unroll 1
  for (uint32_t half = 0; half < cnt; half += 32) {
    const uint32_t fl = half + (uint32_t)lane < cnt ? ctl[half + lane].flags : 0u;
    const uint32_t applied = __ballot_sync(0xFFFFFFFFu, (fl & kApplied) != 0);
    const uint32_t random = __ballot_sync(0xFFFFFFFFu, (fl & kRandom) != 0);
    const uint32_t improved = __ballot_sync(0xFFFFFFFFu, (fl & EG_UPD_IMPROVED) != 0);
    if (!(applied | random | improved)) continue;
    const uint32_t boost_sat = __ballot_sync(0xFFFFFFFFu, (fl & (DEFICIT ? EG_UPD_D_BOOST_SAT : EG_UPD_BOOST_SAT)) != 0);
    const uint32_t pen_kill = __ballot_sync(0xFFFFFFFFu, (fl & (DEFICIT ? EG_UPD_D_PEN_KILL : EG_UPD_PEN_KILL)) != 0);
    const uint32_t mild_kill = __ballot_sync(0xFFFFFFFFu, (fl & (DEFICIT ? EG_UPD_D_PEN_KILL : EG_UPD_MILD_KILL)) != 0);
    const uint32_t proper = __ballot_sync(0xFFFFFFFFu, (fl & (DEFICIT ? EG_UPD_D_PROPER : EG_UPD_PROPER)) != 0);
#pragma unroll 1
    for (uint32_t g = 0; g < 32; g += kGroup) {
      const uint32_t ga = (applied >> g) & 0xFFu, gr = (random >> g) & 0xFFu, gi = (improved >> g) & 0xFFu;
      if (!(ga | gr | gi)) continue;
      const uint32_t j0 = half + g;  // episodes past the end of a short tile have no flags: their operands are never used
      int m[kGroup];
      double f[kGroup], boost[kGroup], pen[kGroup], mild[kGroup];
#pragma unroll
      for (int u = 0; u < kGroup; u++) {
        m[u] = my_rows[(j0 + u) * EG_UPD_ROW];
        f[u] = any_random ? my_fac[(j0 + u) * EG_UPD_ENTRIES] : 1.0;
        boost[u] = DEFICIT ? ctl[j0 + u].d_boost : ctl[j0 + u].boost;
        pen[u] = DEFICIT ? ctl[j0 + u].d_penalty : ctl[j0 + u].penalty;
        mild[u] = DEFICIT ? 1.0 : ctl[j0 + u].mild;
      }
      if (!gi) {
        // No best-strategy change inside the group (all but a handful of groups). Which steps apply to this entry is settled
        // before the multiplications start, as bit masks over the group's eight episodes: boost where the episode's contrast
        // applied and the best strategy holds the entry, penalty where it applied and the count is non-zero, "more than once"
        // where a second multiplication may follow. Every step is then computed and kept or dropped by ONE select on a mask
        // bit, so the only thing a step waits for is the entry's value; the repeat handling is compiled into a second copy of
        // the loop that a warp enters only if one of its lanes has a repeat in this group.
        const bool in_best = occ != 0;
        uint32_t pen_mask = 0u, rep_pen = 0u;
        double pf[kGroup];
#pragma unroll
        for (int u = 0; u < kGroup; u++) {
          pen_mask |= (uint32_t)(m[u] != 0) << u;
          rep_pen |= (uint32_t)(m[u] > 1) << u;
          pf[u] = (!DEFICIT && in_best) ? mild[u] : pen[u];
        }
        const uint32_t boost_mask = in_best ? ga : 0u;
        pen_mask &= ga;
        // a repeat can only matter when the first multiplication does not already end at the fixed point; that it does is
        // known per episode (ctl flags) for every entry inside the clamp range
        // (inside the range now, and every factor applied in this group keeps it there)
        const bool in_range = w >= egrule::kMinWeight && w <= egrule::kMaxWeight && (ga & ~((proper >> g) & 0xFFu)) == 0u;
        const uint32_t gs = (boost_sat >> g) & 0xFFu, gk = (((!DEFICIT && in_best) ? mild_kill : pen_kill) >> g) & 0xFFu;
        rep_pen &= in_range ? (ga & ~gk) : ga;
        const uint32_t rep_boost = occ > 1 ? (in_range ? (ga & ~gs) : ga) : 0u;
        if (!__any_sync(0xFFFFFFFFu, (rep_boost | rep_pen) != 0u)) {
#pragma unroll
          for (int u = 0; u < kGroup; u++) {
            const double tb = w * boost[u];
            const double wb = (egrule::kMaxWeight < tb) ? egrule::kMaxWeight : tb;     // std::min(t, MAX_WEIGHT)
            w = ((boost_mask >> u) & 1u) ? wb : w;
            const double tp = w * pf[u];
            const double wp = (tp >= egrule::kMinWeight) ? tp : egrule::kMinWeight;     // f64::max(t, MIN_WEIGHT), NaN -> MIN_WEIGHT (quirk Q9)
            w = ((pen_mask >> u) & 1u) ? wp : w;
            const double tr = w * f[u];   // std::min(std::max(t, MIN_WEIGHT), MAX_WEIGHT) with both comparisons on t itself
            const double wr = (tr < egrule::kMinWeight) ? egrule::kMinWeight : ((egrule::kMaxWeight < tr) ? egrule::kMaxWeight : tr);
            w = ((gr >> u) & 1u) ? wr : w;
          }
        } else {
#pragma unroll
          for (int u = 0; u < kGroup; u++) {
            const double tb = w * boost[u];
            const double wb = (egrule::kMaxWeight < tb) ? egrule::kMaxWeight : tb;
            w = ((boost_mask >> u) & 1u) ? wb : w;
            // further occurrences in the best strategy: only while they still change the value (MAX_WEIGHT is a fixed point)
            if (((rep_boost >> u) & 1u) && !(w == egrule::kMaxWeight && boost[u] >= 1.0)) w = walk_boost(w, boost[u], occ - 1);
            int mm = m[u];
            if (((rep_pen >> u) & 1u) && mm == 255) mm = walk_recount<DEFICIT>(trajs + first + j0 + u, y, key, rp, cur);  // more than the byte holds
            const double tp = w * pf[u];
            const double wp = (tp >= egrule::kMinWeight) ? tp : egrule::kMinWeight;
            w = ((pen_mask >> u) & 1u) ? wp : w;
            if (((rep_pen >> u) & 1u) && !(w == egrule::kMinWeight && !(pf[u] > 1.0))) w = walk_penalty(w, pf[u], mm - 1);
            const double tr = w * f[u];
            const double wr = (tr < egrule::kMinWeight) ? egrule::kMinWeight : ((egrule::kMaxWeight < tr) ? egrule::kMaxWeight : tr);
            w = ((gr >> u) & 1u) ? wr : w;
          }
        }
        continue;
      }
#pragma unroll
      for (int u = 0; u < kGroup; u++) {
        if (ga & (1u << u)) {
          if (occ && (w != egrule::kMaxWeight || boost[u] < 1.0)) w = walk_boost(w, boost[u], occ);
          if (m[u]) {
            int mm = m[u];
            if (mm == 255) mm = walk_recount<DEFICIT>(trajs + first + j0 + u, y, key, rp, cur);  // more than the byte holds
            const double p = (!DEFICIT && occ) ? mild[u] : pen[u];
            if (mm == 1) w = egrule::max_nan(w * p, egrule::kMinWeight);
            else w = walk_penalty(w, p, mm);
          }
        }
        if (gr & (1u << u)) w = egrule::apply_random_factor(w, f[u]);
        if (gi & (1u << u)) {  // update_best_strategy: best_weights = weights.clone(), the best lists become this episode's
          if (!DEFICIT && live) b.state->best_w[y][key] = w;
          cur = b.slots + first + j0 + u + 1;
          occ = walk_occurrences<DEFICIT>(cur, y, key);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(kWalkThreads) upd_walk_kernel(const eg_traj* trajs, uint32_t n, uint32_t replay, EgUpdBuffers b) {
  extern __shared__ __align__(128) unsigned char walk_smem_raw[];
  WalkSmem& sm = *reinterpret_cast<WalkSmem*>(walk_smem_raw);
  const int y = blockIdx.x, tid = threadIdx.x;
  const bool regular = tid < EG_N_ACTIONS;
  const bool deficit = tid >= 64 && tid < 64 + EG_N_DEFICIT_KEYS;
  const int key = regular ? tid : deficit ? tid - 64 : 0;
  EgUpdState* st = b.state;
  const bool any_random = st->pass_any_random != 0;
  const uint32_t n_tiles = (n + kWalkTile - 1) / kWalkTile;
  const unsigned char* g_ctl = (const unsigned char*)b.ctl;
  const unsigned char* g_cnt = b.counts + (size_t)y * EG_UPD_CHUNK * EG_UPD_ROW;
  const unsigned char* g_fac = (const unsigned char*)(b.factors + (size_t)y * EG_UPD_CHUNK * EG_UPD_ENTRIES);
  constexpr uint32_t kFacBytes = EG_UPD_ENTRIES * sizeof(double);
  auto issue = [&](uint32_t tile, int stage) {  // thread 0 only
    const uint32_t first = tile * kWalkTile, cnt = min((uint32_t)kWalkTile, n - first);
    const uint32_t bar = smem_addr(&sm.full[stage]);
    mbar_expect_tx(bar, cnt * ((uint32_t)(kCtlBytes + EG_UPD_ROW) + (any_random ? kFacBytes : 0u)));
    bulk_g2s(smem_addr(sm.ctl[stage]), g_ctl + (size_t)first * kCtlBytes, cnt * (uint32_t)kCtlBytes, bar);
    bulk_g2s(smem_addr(sm.cnt[stage]), g_cnt + (size_t)first * EG_UPD_ROW, cnt * (uint32_t)EG_UPD_ROW, bar);
    if (any_random) bulk_g2s(smem_addr(sm.factors[stage]), g_fac + (size_t)first * kFacBytes, cnt * kFacBytes, bar);
  };
  if (tid == 0) {
    for (int s = 0; s < kWalkStages; s++) mbar_init(smem_addr(&sm.full[s]), 1u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (uint32_t s = 0; s < (uint32_t)kWalkStages && s < n_tiles; s++) issue(s, (int)s);
  }
  // this thread's entry and how often the current best strategy holds it
  double w = regular ? st->w[y][key] : deficit ? st->dw[y][key] : 0.0;
  const EgUpdSlot* cur = b.slots;  // slot 0: the strategy the pass starts with (all lengths 0 when there is none)
  int occ = 0;
  if (regular) {
    const uint8_t* B = cur->cat + cur->off[y];
    const int LB = cur->len_run[y] + cur->len_def[y];
    for (int i = 0; i < LB; i++) occ += (B[i] == key);
  } else if (deficit) {
    const uint8_t* B = cur->cat + cur->off[y] + cur->len_run[y];
    const int LB = cur->len_def[y];
    for (int i = 0; i < LB; i++) occ += (egrule::deficit_key_of_action(B[i]) == key);
  }
  const bool rp = replay != 0;
  __syncthreads();  // barriers initialised before anyone waits on them
  for (uint32_t tile = 0; tile < n_tiles; tile++) {
    const int stage = (int)(tile % kWalkStages);
    const uint32_t parity = (tile / kWalkStages) & 1u;
    const uint32_t bar = smem_addr(&sm.full[stage]);
    while (!mbar_try_wait(bar, parity)) {}
    const uint32_t first = tile * kWalkTile, cnt = min((uint32_t)kWalkTile, n - first);
    const EgUpdCtl* ctl = (const EgUpdCtl*)sm.ctl[stage];
    // warps 0-1 hold the action entries (threads 61-63 walk entry 0 without storing), warp 2 the deficit entries
    if (tid < 64) walk_tile<false>(ctl, sm.cnt[stage], sm.factors[stage], cnt, first, y, key, regular, rp, any_random, trajs, b, w, occ, cur);
    else walk_tile<true>(ctl, sm.cnt[stage], sm.factors[stage], cnt, first, y, key, deficit, rp, any_random, trajs, b, w, occ, cur);
    __syncthreads();  // everyone is done with this stage
    if (tid == 0 && tile + kWalkStages < n_tiles) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(tile + kWalkStages, stage);
    }
  }
  if (regular) st->w[y][key] = w;
  else if (deficit) st->dw[y][key] = w;
}

// ---- 7. the strategy the next pass starts with --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) upd_carry_kernel(EgUpdBuffers b) {
  const int last = b.state->pass_last_improver;
  if (last < 0) return;
  const unsigned long long* src = (const unsigned long long*)(b.slots + last + 1);
  unsigned long long* dst = (unsigned long long*)b.slots;
  for (int i = threadIdx.x; i < (int)(sizeof(EgUpdSlot) / 8); i += blockDim.x) dst[i] = src[i];
}

}  // namespace

cudaError_t eg_launch_update_pass(const EgUpdBuffers& b, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n, uint32_t base,
                                  uint32_t replay, uint64_t rng_seed, cudaStream_t stream, int* launches) {
  if (launches) *launches = 0;
  if (n == 0) return cudaSuccess;
  if (n > EG_UPD_CHUNK) return cudaErrorInvalidValue;
  upd_score_kernel<<<(n + 255) / 256, 256, 0, stream>>>(d_results, n, b.score, b.state);
  upd_scan_kernel<<<1, 1024, 0, stream>>>(d_results, n, base, b);
  upd_ctl_kernel<<<(n + 127) / 128, 128, 0, stream>>>(n, b);
  upd_expand_kernel<<<(n + 7) / 8, 256, 0, stream>>>(d_trajs, n, replay, b);
  upd_prep_kernel<<<(n + kPrepWarps - 1) / kPrepWarps, kPrepWarps * 32, 0, stream>>>(d_trajs, n, replay, b);
  {
    const uint64_t threads = (uint64_t)n * EG_NY * EG_UPD_ENTRIES;
    upd_random_kernel<<<(uint32_t)((threads + 255) / 256), 256, 0, stream>>>(n, (uint32_t)rng_seed, (uint32_t)(rng_seed >> 32), b);
  }
  static bool smem_opted = false;  // per process; the attribute is per function and device-wide settings are idempotent
  if (!smem_opted) {
    cudaError_t e = cudaFuncSetAttribute(upd_walk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WalkSmem));
    if (e != cudaSuccess) return e;
    smem_opted = true;
  }
  upd_walk_kernel<<<EG_NY, kWalkThreads, sizeof(WalkSmem), stream>>>(d_trajs, n, replay, b);
  upd_carry_kernel<<<1, 256, 0, stream>>>(b);
  if (launches) *launches = 8;
  return cudaGetLastError();
}
