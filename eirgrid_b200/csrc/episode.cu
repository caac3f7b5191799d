// episode.cu — the batched 2025-2050 episode kernel (sm_100a), one episode per WARP.
//
// Replaces, for n episodes at once, the body of the reference's rayon closure up to the write lock:
//   run_iteration / run_simulation / handle_power_deficit      core/iteration.rs:10-95, core/simulation.rs:22-522
//   apply_action / Map::add_generator / add_carbon_offset       core/actions.rs:40-204, utils/map_handler.rs:553-811
//   find_best_generator_location -> find_suitable_location      map_handler.rs:1084-1143, gpu/metal_location_search.rs:110-176
//   Map totals, opinion, capital cost, yearly metrics           map_handler.rs:813-985, analysis/metrics_calculation.rs:7-175
//   sample_action / sample_deficit_action / sample_additional   ai/learning/weights/sampling.rs:76-528
//   update_weights / update_deficit_weights (episode-local)     weights/learning.rs:21-88, weights/deficit.rs:82-135
//   score_metrics                                               ai/metrics/scoring.rs:5-45
//
// Design (DESIGN.md §4.1).
//  * Every float sum/product of the reference runs over Vec<Generator> in insertion order with the pre-existing
//    plants first. The warp keeps the episode's scalar state replicated in every lane (uniform control flow) and adds
//    terms in that same order, so roundings are the reference's; the existing-plant prefix of each accumulator and
//    everything needing pow/exp is tabulated per year on the host. Per-plant TERMS are computed 32 at a time across
//    the lanes, staged in shared memory and folded in sequentially from broadcast reads.
//  * Episode state that is indexed dynamically lives in shared memory, one slice per warp, addressed through the
//    shared window (LDS/STS, never generic loads): the list of plants and offsets built so far and this year's private
//    copy of the weight rows.
//  * The 100x100 placement scan becomes a walk, 32 candidates per step, down a per-(class, year) list of sites sorted
//    by static score (the score when no simulation-built plant is in range). A plant in range can only lower a site's
//    score (all factors < 1, rounding is monotone), so the walk stops once static scores fall below the best exact
//    score found. Every site still in the race multiplies the factors of the plants in its range in plant order, one
//    site per lane: the squared cell distance is ONE dot-product instruction per (site, plant) (|s|^2 + |g|^2 - 2 s.g from
//    packed bytes), plant words are read four at a time, and a plant out of range multiplies by a 1.0 stored after the
//    class's factors, so there is no range test and four lookups are in flight (Warp::place). While the walk runs, the
//    episode's running sums wait in shared memory (Warp::stash): 94 registers, 20 warps per SM.
//  * Philox draws are produced 32 at a time (lane l computes draw base+l) and handed out by shuffle.
//  * Compiled with --fmad=false: + - * / sqrt are the reference's IEEE operations, no contraction.
//  * The kernel is bound by instruction fetch as much as by issue: it is instantiated per (REPLAY, GEOM, MODE) so that the
//    training launch runs an image without the optional outputs, the replay-best branches and the sampler it does not use.
#include "episode.cuh"
#include "update_rule.hpp"
#include <algorithm>
#include <cstddef>

extern __shared__ __align__(16) unsigned char smem[];  // dynamic shared memory of the episode kernels: one slice per warp

namespace {

constexpr unsigned kFull = 0xFFFFFFFFu;

// The tuning constants of this file are the measured optimum (profiles/r02_eval_loop.md, r02_ab_candidates.md). An experiment adds
// its own -D switch on a branch and merges only the winner, without the switch. Outputs do not depend on any of them.
constexpr int kEvalUnroll = 2;            // groups of four plants per trip of the placement evaluation loop: 1 and 3 are slower, 4 costs 18 % on the trained table
constexpr int kEvalUnrollStagnation = 1;  // the same in the stagnation-sampler instantiation on compact maps, the larger one: 2 % faster not unrolled
constexpr int kYearStartUnroll = 1;       // year_start's re-sum over the plants: unrolled by 2 or 4, +1 % on the initial table, -1..-3 % trained
constexpr int kFoldUnroll = 2;            // year folds: not unrolled is slower
constexpr int kScanUnroll = 4;            // sequential sampling scans: unrolled by 2 or 1 is slower

// -DEG_DEBUG_BOUNDS: index checks on the shared-memory structures; a violation sets bit 30 of eg_result.flags, which makes
// every parity test fail (compute-sanitizer is not available on the GPU pool). Compiled out otherwise.
#ifdef EG_DEBUG_BOUNDS
#define EG_CHECK(cond) do { if (!(cond)) flags |= 0x40000000u; } while (0)
#else
#define EG_CHECK(cond) do { } while (0)
#endif
constexpr int kBattery100 = 3 * 12;   // AddGenerator(BatteryStorage, 100 %), simulation.rs:376
constexpr int kGasPeaker100 = 3 * 8;  // sampling fallbacks, sampling.rs:185,237,321,377

// ---- per-warp shared-memory slice --------------------------------------------------------------------------
// two buffers of policy rows (year parity): [61 regular | 15 deficit | 21 count weights | pad]; the rows of year y+1 are
// copied in asynchronously (cp.async) while year y runs, the rows of year y are this episode's private, editable copy
constexpr int kRowDoubles = EG_N_ACTIONS + EG_N_DEFICIT_KEYS + EG_N_COUNT_KEYS + 1;  // 98
constexpr int kRowBytes = 8 * kRowDoubles;
constexpr int kOffRows = 0;
constexpr int kOffScratch = kOffRows + 2 * kRowBytes;           // double2[32] fold staging | double[61] + uint8[64] sorted row
constexpr int kScratchBytes = 8 * EG_N_ACTIONS + 64;            // 552 >= 512
constexpr int kOffSortIdx = kOffScratch + 8 * EG_N_ACTIONS;     // uint8[64] (inside the scratch area)
constexpr int kOffVars = (kOffScratch + kScratchBytes + 15) & ~15;  // double[32]  rarely used episode scalars (kV*)
constexpr int kOffGxy = kOffVars + 8 * 32;                      // uint32[EG_MAX_NEW_GENERATORS] plant words: cell (gi << 8) | gj in the low half,
                                                                // gi*gi + gj*gj as (q & 63) << 16 | (q >> 6) << 24 in the high half (compact maps)
constexpr int kOffGat = kOffGxy + 4 * EG_MAX_NEW_GENERATORS;    // uint16[EG_MAX_NEW_GENERATORS] type(4) mult(2) build(5)
constexpr int kOffOffs = kOffGat + 2 * EG_MAX_NEW_GENERATORS;   // uint16[EG_MAX_OFFSETS]
constexpr int kOffCounts = kOffOffs + 2 * EG_MAX_OFFSETS;       // uint16[26] deficit + uint16[26] additional recorded per year
constexpr int kSliceBytes = (kOffCounts + 4 * EG_NY + 15) & ~15;  // 6,896 B per warp
static_assert(kOffScratch % 16 == 0 && kOffVars % 8 == 0 && kOffGxy % 16 == 0 && EG_MAX_NEW_GENERATORS % 4 == 0 && kOffOffs % 4 == 0 && kOffCounts % 4 == 0, "alignment");
// a plant word no site is in range of (cell (0, 0), squared norm 8191): pads the plant list to a multiple of four on compact maps
constexpr uint32_t kPlantSentinel = (63u << 16) | (127u << 24);
// the action record (eg_traj / eg_sites) is written straight to global memory, one slot per recorded action (lane 0), the
// unused tail once at the end of the episode with 8-byte stores
static_assert(offsetof(eg_traj, actions) % 8 == 0 && sizeof(eg_traj) % 8 == 0 && EG_TRAJ_CAPACITY % 8 == 0 && sizeof(eg_sites) % 8 == 0, "tail fill uses 8-byte stores");

// slots of the per-warp scalar area: values every lane agrees on that are touched a few times per year
enum { kVTotalCost = 0, kVTotalCredit, kVTotalSales, kVGcostPrev, kVOcostPrev, kVLwTotal, kVInitNet, kVInitOpinion, kVInitBalance, kVInitCost, kVScaledTotal, kVStash /* 13 slots */ };

// ---- Philox4x32-10, counter = (episode lo, episode hi, draw, stream 0), key = seed ------------------------
__device__ __noinline__ unsigned long long philox_u64(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2) {
  uint32_t c3 = 0u;
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return (unsigned long long)c0 | ((unsigned long long)c1 << 32);
}

// IEEE-754 double division (correctly rounded, like the reference's `/`). One out-of-line copy: the kernel is bound
// by instruction fetch, and ~20 inlined division sequences were a fifth of its hot code.
__device__ __noinline__ double ddiv(double a, double b) { return a / b; }

struct State {  // ActionResult, ai/metrics/simulation_metrics.rs:14-19
  double net, opinion, balance, cost;
};

// evaluate_action_impact(.., None), scoring.rs:60-84
__device__ __forceinline__ double action_impact(const State& cur, const State& nw) {
  if (cur.net > 0.0) {
    // a plant without CO2 leaves the emissions unchanged: +0 / x = +0, without the division (whose hardware sequence
    // takes its ~100-instruction slow path for a zero numerator)
    const double reduction = cur.net - nw.net;
    return reduction == 0.0 ? reduction : ddiv(reduction, fmax(fabs(cur.net), 1.0));
  }
  double cost_change = nw.cost - cur.cost;
  double cost_improvement = ddiv(-cost_change, fmax(fabs(cur.cost), 1.0));
  double opinion_improvement = ddiv(nw.opinion - cur.opinion, fmax(fabs(cur.opinion), 1.0));
  double cost_weight = cur.cost > egrule::kMaxCost * 8.0 ? 0.8 : 0.5;
  double opinion_weight = 1.0 - cost_weight;
  return cost_improvement * cost_weight + opinion_improvement * opinion_weight;
}

__device__ __forceinline__ double shfl_f64(double v, int src) { return __shfl_sync(kFull, v, src); }

// plant attributes: type(4) mult(2) build(5); plant cells use the byte order of the `order` table, (i << 8) | j
__device__ __forceinline__ uint32_t pack_attr(int t, int m, int b) { return (uint32_t)t | ((uint32_t)m << 4) | ((uint32_t)b << 6); }

// read-only table in shared memory addressed by a 32-bit shared-window address (kept in a register by the caller)
__device__ __forceinline__ double lds_f64(uint32_t addr) {
  double v;
  asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}

// c + (low half of a as s16) * (byte 0 of b) + (high half of a as s16) * (byte 1 of b), bytes unsigned
__device__ __forceinline__ int dp2a_lo_su(uint32_t a, uint32_t b, int c) {
  int d;
  asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// walk-list entries are read once per placement step and never again: they stream past the L1 (`LDG.E.NA`, no allocation), which
// keeps it for the tables that are re-read (type, year and plant terms, site opinions, policy constants): +1 % / +1.8 % (initial /
// trained table, profiles/r02_eval_loop.md)
__device__ __forceinline__ double2 ldg_stream(const double2* p) {
  double2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ int ldg_stream(const uint16_t* p) {
  unsigned short v;
  asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(v) : "l"(p));
  return (int)v;
}

// keeps a value in a register: the compiler may not re-derive it from its definition inside the hot loops
__device__ __forceinline__ uint32_t opaque(uint32_t v) {
  asm volatile("" : "+r"(v));
  return v;
}

// sampling.rs:445-490 / 492-528: the fixed fallback tables (replay mode without a stored action)
__device__ __noinline__ int smart_fallback_pick(int y, uint32_t choice) {
  const int year = EG_BASE_YEAR + y;
  const uint32_t storage = year < 2035 ? 10 : 20;
  const uint32_t offset = year < 2035 ? 5 : (year < 2045 ? 15 : 25);
  const uint32_t gas = year < 2035 ? 15 : (year < 2045 ? 10 : 5);
  if (choice < 15) return 3 * 0;
  choice -= 15;
  if (choice < 10) return 3 * 1;
  choice -= 10;
  if (choice < 15) return 3 * 4;
  choice -= 15;
  if (choice < storage) return 3 * 12;
  choice -= storage;
  if (choice < offset) return 45 + 3 * 0;
  choice -= offset;
  if (choice < offset) return 45 + 3 * 2;
  choice -= offset;
  if (choice < gas) return 3 * 7;
  return kBattery100;
}
__device__ __forceinline__ uint32_t smart_fallback_total(int y) {
  const int year = EG_BASE_YEAR + y;
  return 40u + (year < 2035 ? 10u : 20u) + 2u * (year < 2035 ? 5u : (year < 2045 ? 15u : 25u)) + (year < 2035 ? 15u : (year < 2045 ? 10u : 5u));
}
__device__ __noinline__ int smart_deficit_fallback_pick(uint32_t choice) {  // ((0.07*0.5) as u32 == 0, (0.06*0.5*100) as u32 == 3)
  if (choice < 30) return 3 * 8;
  choice -= 30;
  if (choice < 30) return 3 * 12;
  choice -= 30;
  if (choice < 20) return 3 * 7;
  choice -= 20;
  if (choice < 10) return 3 * 0;
  choice -= 10;
  if (choice < 3) return 3 * 4;
  return kBattery100;
}

// stagnation branch of sample_action (sampling.rs:190-220) for rows edited in this episode: stable descending
// sort by rank counting and the powers, both spread over the lanes
__device__ __noinline__ void sort_local(uint32_t sb, uint32_t sb_rows, int lane, double power) {
  const double* lw = (const double*)(smem + sb_rows);
  double* scaled = (double*)(smem + sb + kOffScratch);
  uint8_t* sort_idx = smem + sb + kOffSortIdx;
  for (int k = lane; k < EG_N_ACTIONS; k += 32) {
    const double wk = lw[k];
    int rank = 0;
    for (int j = 0; j < EG_N_ACTIONS; j++) {
      const double wj = lw[j];
      rank += (wj > wk) || (wj == wk && j < k);
    }
    sort_idx[rank] = (uint8_t)k;
    scaled[rank] = pow(wk, power);
  }
  __syncwarp();
}

// deficit key of a generator type (0xF: none) and action code of a key < 14, from the nibble forms of update_rule.hpp
__device__ __forceinline__ int deficit_key_of_type(int t) { return (int)((egrule::kKeyOfType >> (4 * t)) & 0xF); }
__device__ __forceinline__ int deficit_key_action(int k) { return 3 * (int)((egrule::kTypeOfKey >> (4 * k)) & 0xF); }

// MODE 0: every option decided at run time. MODE 1, 2: the training launch — no optional outputs (eg_sites, eg_yearly),
// no replay-best mode, count weights present — with the plain sampler (iterations_without_improvement <= 500) or the
// stagnation sampler (> 500) compiled in alone. EG_OPT(x) is x in the general instantiation and false in the lean ones.
#define EG_OPT(x) (!LEAN && (x))
// GEOM (EgDeviceMap::near_geom): 0 compact map (at most 64 sites per axis), 1 medium (at most 181; blocks of 10 warps around a
// factor table of up to 5,600 entries), 2 general (at most 256 sites per axis, factor table read from global memory).
template <bool REPLAY, int GEOM, int MODE>
struct Warp {
  static constexpr bool WIDE = GEOM == 2;
  static constexpr bool LEAN = MODE != 0;
  __device__ __forceinline__ bool stagnation() const { return MODE == 0 ? p.policy->iwi > 500 : MODE == 2; }
  const EgEpisodeParams& p;
  const EgSmallTables* __restrict__ T;
  const int lane;
  const uint32_t sb;  // byte offset of this warp's slice in the block's dynamic shared memory
  // warp-uniform episode state (identical in every lane)
  double gen0, gen1, gen2;    // plain / intermittent / storage generation accumulators
  double co2, op_sum;
  double gcost, ocost;        // capital cost of new plants / offsets re-priced at the current year (map_handler.rs:955-962);
                              // the same sums re-priced at year-1 live in the scalar area (kVGcostPrev, kVOcostPrev)
  double off_amount;          // calc_total_carbon_offset(year)
  uint32_t n_gens, n_offs, flags;
  uint32_t ep;                // index of the episode in the batch (output slot)
  uint32_t rec_used;          // slots of the action record written so far (all years)
  bool rows_dirty, dw_dirty, sorted_valid, total_valid;
  bool folded;                // this year's plant/offset sums (op_sum, gcost, ocost, off_amount) are valid
  // Philox: lane l holds draw number rbase + l of episode `rng_id`
  unsigned long long rng_id;
  uint32_t draw, rbase;
  unsigned long long rbuf;

  __device__ Warp(const EgEpisodeParams& p_, uint32_t sb_, int lane_) : p(p_), T(p_.map.small), lane(lane_), sb(sb_) {}

  __device__ __forceinline__ double* VARS() const { return (double*)(smem + sb + kOffVars); }
  __device__ __forceinline__ uint32_t* GXY() const { return (uint32_t*)(smem + sb + kOffGxy); }
  __device__ __forceinline__ uint16_t* GAT() const { return (uint16_t*)(smem + sb + kOffGat); }

  __device__ __forceinline__ double* LW(int y) const { return (double*)(smem + sb + kOffRows + (y & 1) * kRowBytes); }
  __device__ __forceinline__ double* LDW(int y) const { return LW(y) + EG_N_ACTIONS; }
  __device__ __forceinline__ double* LCW(int y) const { return LW(y) + EG_N_ACTIONS + EG_N_DEFICIT_KEYS; }
  __device__ __forceinline__ double2* SCR() const { return (double2*)(smem + sb + kOffScratch); }
  __device__ __forceinline__ uint16_t* OFFS() const { return (uint16_t*)(smem + sb + kOffOffs); }
  __device__ __forceinline__ uint16_t* COUNTS() const { return (uint16_t*)(smem + sb + kOffCounts); }


  // ---- random draws ---------------------------------------------------------------------------------------
  __device__ __forceinline__ unsigned long long u64() {
    uint32_t off = draw - rbase;
    if (off >= 32u) {
      rbase = draw;
      rbuf = philox_u64((uint32_t)p.seed, (uint32_t)(p.seed >> 32), (uint32_t)rng_id, (uint32_t)(rng_id >> 32), draw + (uint32_t)lane);
      off = 0;
    }
    draw++;
    return __shfl_sync(kFull, rbuf, (int)off);
  }
  __device__ __forceinline__ double f64() { return (double)(u64() >> 11) * (1.0 / 9007199254740992.0); }
  __device__ __forceinline__ uint32_t index(uint32_t n) { return (uint32_t)__umul64hi(u64(), (unsigned long long)n); }

  // (cost-opinion term, get_current_cost) of a simulation-built plant in year y: one 16-byte read of the host table
  // (base_cost * inflation * technology_factor * location_modifier * multiplier, const_funcs.rs:56, generator.rs:593)
  __device__ __forceinline__ double2 plant_terms(int t, int m, int b, int y) const {
    return __ldg((const double2*)p.map.plant_terms + EG_OPC_INDEX(y, t, m, b));
  }
  __device__ __forceinline__ double gen_cost(int t, int m, int b, int y) const { return plant_terms(t, m, b, y).y; }
  __device__ __forceinline__ double off_cost(int o, int m, int y) const {
    return __ldg(&T->off_base_cost[o]) * __ldg(&T->year[y].inflation) * __ldg(&T->mult[m]);  // carbon_offset.rs:188-195
  }
  __device__ __forceinline__ double gen_opinion(int site, int t, int y, double cost_term) const {
    // calc_new_generator_opinion, map_handler.rs:946-948
    return 0.03 * __ldg(&p.map.site_opinion[site]) + __ldg(&T->op_type[y][t]) + cost_term;
  }

  // Start of a year: re-fold the per-plant terms that depend on the year, in plant order (the order of the
  // reference's iterator sums). Terms are computed one plant per lane, staged in shared memory and added
  // sequentially from broadcast reads.
  //  * capital cost re-priced at year-1 over this year's fleet continues last year's sum (the plants built this year
  //    are appended to it), so it is carried, not recomputed;
  //  * generation and CO2 of a simulation-built plant do not depend on the year: those sums are re-folded only when
  //    the existing-plant prefix changed (the years the pre-existing fleet comes online, quirk Q1).
  __device__ __forceinline__ void year_start(int y) {
    const EgYearRow& yr = T->year[y];
    if (y == 0 || __ldg(&yr.prefix_changed) != 0) {
      gen0 = __ldg(&yr.ex_gen[0]); gen1 = __ldg(&yr.ex_gen[1]); gen2 = __ldg(&yr.ex_gen[2]);
      co2 = __ldg(&yr.ex_co2);
      const uint16_t* gat = GAT();
#pragma unroll kYearStartUnroll
      for (uint32_t i = 0; i < n_gens; i++) {
        const int t = gat[i] & 0xF;
        // (plain, intermittent, storage, CO2) of the type: adding +0.0 leaves the other accumulators unchanged bit for bit
        const double2 s01 = __ldg((const double2*)&T->type_sums[t][0]), s23 = __ldg((const double2*)&T->type_sums[t][2]);
        gen0 += s01.x; gen1 += s01.y; gen2 += s23.x;
        co2 += s23.y;
      }
    }
  }

  // The year-dependent sums over the episode's plants and offsets (opinion, capital cost, offset amount and cost). They are
  // read only by the deficit handler's state evaluations, by the yearly-metrics output and by the 2050 result, so the
  // episode re-folds them only in years that need them: every fold starts from the tabulated prefix and runs over the whole
  // list in order, so skipping a year changes nothing in the years that do fold.
  __device__ __forceinline__ void year_folds(int y) {
    const EgYearRow& yr = T->year[y];
    op_sum = __ldg(&yr.ex_opinion_sum);
    if (lane == 0) { VARS()[kVGcostPrev] = gcost; VARS()[kVOcostPrev] = ocost; }
    gcost = 0.0;
    const int n = p.map.grid_n;
    double2* scr = SCR();
    for (uint32_t base = 0; base < n_gens; base += 32) {
      const uint32_t i = base + lane;
      if (i < n_gens) {
        const uint32_t xy = GXY()[i], at = GAT()[i];
        const int gj = xy & 0xFF, gi = (xy >> 8) & 0xFF, t = at & 0xF, m = (at >> 4) & 0x3, b = at >> 6;
        EG_CHECK(t < EG_NT && m < EG_N_MULTS && b <= y && gi < n && gj < n);
        const double2 pt = plant_terms(t, m, b, y);
        scr[lane] = make_double2(gen_opinion(gi * n + gj, t, y, pt.x), pt.y);
      }
      __syncwarp();
      const int cnt = min(32u, n_gens - base);
#pragma unroll kFoldUnroll
      for (int j = 0; j < cnt; j++) {
        const double2 v = scr[j];
        op_sum += v.x;
        gcost += v.y;
      }
      __syncwarp();
    }
    ocost = 0.0; off_amount = 0.0;
    for (uint32_t base = 0; base < n_offs; base += 32) {
      const uint32_t i = base + lane;
      if (i < n_offs) {
        const uint32_t o = OFFS()[i];
        const int ot = o & 3, m = (o >> 2) & 3, b = (o >> 4) & 0x1F;
        EG_CHECK(b <= y && y - b < EG_NY);
        const double maturity = __ldg(&T->natural_offset[ot]) ? __ldg(&T->maturity[y - b]) : 1.0;
        scr[lane] = make_double2(__ldg(&T->off_amount[ot]) * maturity, off_cost(ot, m, y));
      }
      __syncwarp();
      const int cnt = min(32u, n_offs - base);
#pragma unroll kFoldUnroll
      for (int j = 0; j < cnt; j++) {
        const double2 v = scr[j];
        off_amount += v.x;
        ocost += v.y;
      }
      __syncwarp();
    }
  }

  // the episode's running sums and the deficit handler's current state wait in shared memory while the placement walk runs, so the
  // walk has their 26 registers
  __device__ __forceinline__ void stash(const State& cur, double remaining) {
    if (lane == 0) {
      double* v = VARS() + kVStash;
      v[0] = gen0; v[1] = gen1; v[2] = gen2; v[3] = co2; v[4] = op_sum; v[5] = gcost; v[6] = ocost; v[7] = off_amount;
      v[8] = cur.net; v[9] = cur.opinion; v[10] = cur.balance; v[11] = cur.cost; v[12] = remaining;
    }
    __syncwarp();
  }
  __device__ __forceinline__ double lds_v(uint32_t addr) const {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
  }
  __device__ __forceinline__ void unstash(State& cur, double& remaining) {
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(smem) + sb + kOffVars + 8u * kVStash;
    gen0 = lds_v(a); gen1 = lds_v(a + 8); gen2 = lds_v(a + 16); co2 = lds_v(a + 24); op_sum = lds_v(a + 32); gcost = lds_v(a + 40);
    ocost = lds_v(a + 48); off_amount = lds_v(a + 56);
    cur.net = lds_v(a + 64); cur.opinion = lds_v(a + 72); cur.balance = lds_v(a + 80); cur.cost = lds_v(a + 88); remaining = lds_v(a + 96);
    __syncwarp();  // every lane has its copy before lane 0 may write the slots again
  }
  __device__ __forceinline__ State state(int y) const {  // simulation.rs:122-135
    State s;
    s.net = co2 - off_amount;
    const uint32_t cnt = __ldg(&T->year[y].ex_active) + n_gens;
    s.opinion = cnt > 0 ? ddiv(op_sum, (double)cnt) : 1.0;
    s.balance = (gen0 + gen1 + gen2) - __ldg(&T->year[y].usage_total);
    s.cost = gcost + ocost;
    return s;
  }

  // MetalLocationSearch::find_suitable_location (CPU branch) as a 32-wide walk down the pre-sorted site list. Returns the
  // winning cell as (i << 8) | j (the order of these words is the scan order of the sites), -1 when no site scores above 0.
  __device__ __forceinline__ int place(int t, int y) {
    EG_CHECK(t >= 0 && t < EG_NT);
    // everything the walk needs to know about the type, one 8-byte read: placement class, radius class, water flag and first
    // entry of the class in the block-shared factor table | first squared cell distance outside the penalty radius
    const uint2 info = __ldg((const uint2*)&T->place_info[t][0]);
    const int pc = info.x & 0xF, rc = (info.x >> 4) & 0xF;
    EG_CHECK(pc < EG_N_PCLASS && rc < EG_N_RCLASS);
    const bool water = (info.x & 0x100u) != 0;
    const int nf_off = (int)(info.x >> 16);
    const int r2lim = (int)info.y;  // cell offsets with d2 < r2lim are inside the penalty radius
    const int ns = p.map.n_sites, n = p.map.grid_n;
    const size_t base = ((size_t)pc * EG_NY + y) * ns + lane;
    // this lane's entry of the current step; entries past the end of the list read as score 0, which ends the walk
    const uint16_t* __restrict__ op = p.map.order + base;
    const double2* __restrict__ wp = (const double2*)p.map.walk + base;
    int left = ns - lane;  // entries from this lane's position to the end of the list
    // distance/radius by squared cell distance: block-shared copy in shared memory (narrow maps), else global
    // (the block-shared copy sits at the start of the dynamic shared memory)
    const double* __restrict__ nf = p.map.near_factor + rc * p.map.r2_stride;
    const uint32_t nf_base = opaque((uint32_t)__cvta_generic_to_shared(smem));
    const double size_factor = __ldg(&T->size_factor);
    const uint32_t* gw = GXY();
    double best_score = 0.0;
    int best_cell = -1;
    double2 sp_next = make_double2(0.0, 0.0);   // (static score, prefix score)
    int packed_next = 0;                        // (i << 8) | j of the candidate site
    if (left > 0) { sp_next = ldg_stream(wp); packed_next = ldg_stream(op); }
    for (;;) {
      const double s_static = sp_next.x, pre = sp_next.y;
      const int packed = packed_next;
      // every site still in the race is evaluated exactly; zero scores never win
      const bool cand = s_static > 0.0 && !(s_static < best_score);
      // the list is sorted and lane 0 holds the step's highest static score: when lane 0 is out of the race, nothing from
      // here on can beat the best so far
      if ((__ballot_sync(kFull, cand) & 1u) == 0u) break;
      {  // entries of the next step: in flight while this step is examined (requested after the exit test, so that the walk never
         // leaves with a load outstanding — whoever reuses its registers next would wait an L2 round trip for it: +1.7 %)
        left -= 32; wp += 32; op += 32;
        sp_next = make_double2(0.0, 0.0);
        if (left > 0) { sp_next = ldg_stream(wp); packed_next = ldg_stream(op); }
      }
      // survivors multiply their factors in plant order (== multiplication order of the reference), one site per lane
      double sc = pre;
      if (GEOM == 0) {
        // coordinates < 64: |s - g|^2 = |s|^2 + |g|^2 - 2 s.g in ONE IDP.4A per (32 sites x 1 plant): the site's bytes are
        // (-2 sj, -2 si, 1, 64), the plant word's (gj, gi, |g|^2 & 63, |g|^2 >> 6), the accumulator |s|^2 (+ the offset of
        // the class's factors in the block-shared table, so that the sum addresses the table directly). Four plant words per
        // 16-byte broadcast read; the list is padded to a multiple of four with words no site is in range of.
        const uint32_t sa = ((0x8080u - 2u * (uint32_t)packed) ^ 0x8080u) | 0x40010000u;
        const int sq = __dp4a(packed, packed, nf_off);
        const uint4* g4 = (const uint4*)gw;
        const uint32_t groups = (n_gens + 3u) >> 2;
        // No predicates: a plant out of range reads the 1.0 that ends the class's factors (x * 1.0 == x bit for bit), so the
        // four lookups of a group are in flight together and only the multiplications wait for each other. (Lanes out of the
        // race multiply along; their result is not looked at.) Measured alternatives, all with identical outputs
        // (profiles/r02_eval_loop.md): predicated lookups as on medium maps (-3.5 % on the shipped map), a two-stage software
        // pipeline, unrolling by 1, 3 and 4, 16 lane-private copies of the table (no bank conflicts, but 3-6 % slower: less L1).
        const int lim = nf_off + r2lim;
        constexpr int kUnroll = MODE == 2 ? kEvalUnrollStagnation : kEvalUnroll;
#pragma unroll kUnroll
        for (uint32_t q = 0; q < groups; q++) {
          const uint4 w4 = g4[q];
          const int d0 = min(__dp4a((int)sa, (int)w4.x, sq), lim), d1 = min(__dp4a((int)sa, (int)w4.y, sq), lim);
          const int d2 = min(__dp4a((int)sa, (int)w4.z, sq), lim), d3 = min(__dp4a((int)sa, (int)w4.w, sq), lim);
          EG_CHECK(d0 >= nf_off && d1 >= nf_off && d2 >= nf_off && d3 >= nf_off);
          const double f0 = lds_f64(nf_base + 8u * (uint32_t)d0), f1 = lds_f64(nf_base + 8u * (uint32_t)d1);
          const double f2 = lds_f64(nf_base + 8u * (uint32_t)d2), f3 = lds_f64(nf_base + 8u * (uint32_t)d3);
          sc *= f0;  // score *= distance / penalty_radius, in plant order
          sc *= f1;
          sc *= f2;
          sc *= f3;
        }
      } else if (GEOM == 1) {
        // up to 181 sites per axis (|g|^2 fits 16 bits): the plant word is cell | |g|^2 << 16, and
        // |s - g|^2 = (|s|^2 - 2 s.g) + |g|^2 is one IDP.2A (16-bit (-2 sj, -2 si) times the word's two low bytes) and one add
        // of the word's high half; same groups of four as on compact maps, but predicated lookups: only the lanes in range read
        // the table, the others multiply by a register 1.0. On the 10x grid the shared-memory pipe is the limiter (97 % busy,
        // half of its wavefronts bank conflicts of the random lookups), and fewer wavefronts are +3.4 % there
        // (profiles/r02_eval_loop.md).
        const int si = packed >> 8, sj = packed & 0xFF;
        const uint32_t sa = ((uint32_t)(-2 * sj) & 0xFFFFu) | ((uint32_t)(-2 * si) << 16);
        const int sq = si * si + sj * sj + nf_off;
        const uint4* g4 = (const uint4*)gw;
        const uint32_t groups = (n_gens + 3u) >> 2;
        const int lim = nf_off + r2lim;
#pragma unroll kEvalUnroll
        for (uint32_t q = 0; q < groups; q++) {
          const uint4 w4 = g4[q];
          const int d0 = dp2a_lo_su(sa, w4.x, sq) + (int)(w4.x >> 16), d1 = dp2a_lo_su(sa, w4.y, sq) + (int)(w4.y >> 16);
          const int d2 = dp2a_lo_su(sa, w4.z, sq) + (int)(w4.z >> 16), d3 = dp2a_lo_su(sa, w4.w, sq) + (int)(w4.w >> 16);
          double f0 = 1.0, f1 = 1.0, f2 = 1.0, f3 = 1.0;
          if (d0 < lim) f0 = lds_f64(nf_base + 8u * (uint32_t)d0);
          if (d1 < lim) f1 = lds_f64(nf_base + 8u * (uint32_t)d1);
          if (d2 < lim) f2 = lds_f64(nf_base + 8u * (uint32_t)d2);
          if (d3 < lim) f3 = lds_f64(nf_base + 8u * (uint32_t)d3);
          sc *= f0;  // score *= distance / penalty_radius, in plant order
          sc *= f1;
          sc *= f2;
          sc *= f3;
        }
      } else {
        const int si = packed >> 8, sj = packed & 0xFF;
#pragma unroll 4
        for (uint32_t g = 0; g < n_gens; g++) {
          const uint32_t pk = gw[g];
          const int dj = sj - (int)(pk & 0xFF), di = si - (int)((pk >> 8) & 0xFF);
          const int d2 = min(di * di + dj * dj, r2lim);
          sc *= __ldg(&nf[d2]);  // the global table holds 1.0 at r2_limit[rc] (host_tables.cpp)
        }
      }
      if (water) sc *= __ldg(&p.map.coast_factor[(packed >> 8) * n + (packed & 0xFF)]);
      sc *= size_factor;
      // strict '>' in scan order: the maximum wins, equal scores keep the lower site. Scores are >= 0, so their
      // high and low words order like the doubles: two 32-bit maximum reductions give the exact maximum.
      const uint32_t hi = cand ? (uint32_t)__double2hiint(sc) : 0u;
      const uint32_t mh = __reduce_max_sync(kFull, hi);
      const uint32_t lo = (cand && hi == mh) ? (uint32_t)__double2loint(sc) : 0u;
      const uint32_t ml = __reduce_max_sync(kFull, lo);
      const int c_cell = (int)__reduce_min_sync(kFull, (cand && hi == mh && lo == ml) ? (uint32_t)packed : 0x7FFFFFFFu);
      const double c_score = __hiloint2double((int)mh, (int)ml);
      if (c_score > best_score || (c_score == best_score && best_cell >= 0 && c_cell < best_cell)) { best_score = c_score; best_cell = c_cell; }
    }
    return best_cell;
  }

  // false: the episode's plant list is full (flagged); nothing was added
  __device__ __forceinline__ bool add_generator(int cell, int t, int m, int y) {
    if (n_gens >= EG_MAX_NEW_GENERATORS) { flags |= EG_FLAG_GEN_OVERFLOW; return false; }
    const int gi = cell >> 8, gj = cell & 0xFF;
    EG_CHECK(gi >= 0 && gi < p.map.grid_n && gj >= 0 && gj < p.map.grid_n && n_gens < EG_MAX_NEW_GENERATORS && t < EG_NT && m < EG_N_MULTS && y < EG_NY);
    {
      // |g|^2 next to the cell: as (q & 63, q >> 6 <= 127) on compact maps, as 16 bits on maps of up to 181 sites per axis
      const uint32_t norm = (uint32_t)(gi * gi + gj * gj);
      const uint32_t word = (uint32_t)cell | (GEOM == 0 ? ((norm & 63u) << 16) | ((norm >> 6) << 24) : (GEOM == 1 ? norm << 16 : 0u));
      uint32_t* gw = GXY();
      if (lane == 0) { gw[n_gens] = word; GAT()[n_gens] = (uint16_t)pack_attr(t, m, y); }
      else if (GEOM != 2 && lane < 4 && (n_gens & 3u) == 0u) gw[n_gens + lane] = GEOM == 0 ? kPlantSentinel : 0xFFFF0000u;  // pads the new group of four
    }
    n_gens++;
    __syncwarp();
    // (plain, intermittent, storage, CO2) of the type: adding +0.0 leaves the other accumulators unchanged bit for bit
    const double2 s01 = __ldg((const double2*)&T->type_sums[t][0]), s23 = __ldg((const double2*)&T->type_sums[t][2]);
    gen0 += s01.x; gen1 += s01.y; gen2 += s23.x;
    co2 += s23.y;
    if (folded) {  // keep this year's folded sums current
      const double2 pt = plant_terms(t, m, y, y);
      op_sum += gen_opinion(gi * p.map.grid_n + gj, t, y, pt.x);
      gcost += pt.y;
      if (y > 0 && lane == 0) VARS()[kVGcostPrev] += gen_cost(t, m, y, y - 1);
    }
    return true;
  }
  __device__ __forceinline__ void add_offset(int ot, int m, int y) {
    if (n_offs >= EG_MAX_OFFSETS) { flags |= EG_FLAG_OFFSET_OVERFLOW; return; }
    if (lane == 0) OFFS()[n_offs] = (uint16_t)(ot | (m << 2) | (y << 4));
    n_offs++;
    __syncwarp();
    if (folded) {  // keep this year's folded sums current
      const double maturity = __ldg(&T->natural_offset[ot]) ? __ldg(&T->maturity[0]) : 1.0;
      off_amount += __ldg(&T->off_amount[ot]) * maturity;
      ocost += off_cost(ot, m, y);
      if (y > 0 && lane == 0) VARS()[kVOcostPrev] += off_cost(ot, m, y - 1);
    }
  }

  // ---- episode-local learning (the deficit handler edits this year's rows of its private weights) ----------
  // asynchronous copy of the policy rows of year y (w[y] | dw[y] | cw[y]) into the buffer of that year's parity
  __device__ __forceinline__ void prefetch_rows(int y) {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem) + sb + kOffRows + (uint32_t)(y & 1) * kRowBytes;
    static_assert(kRowDoubles == EG_POLICY_ROW && kRowBytes % 16 == 0, "the row is copied in 16-byte pieces");
    const char* src = (const char*)&p.policy->rows[y][0];
    for (int k = lane; k < kRowBytes / 16; k += 32)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (uint32_t)k), "l"(src + 16 * k) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  // the rows of year y are complete (requested a year earlier); request those of year y+1
  __device__ __forceinline__ void load_rows(int y) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    if (y + 1 < EG_NY) prefetch_rows(y + 1);
    rows_dirty = false; dw_dirty = false; sorted_valid = false; total_valid = false;
    if (stagnation()) {  // the snapshot's sorted, scaled row of this year (host libm) for the stagnation sampler
      double* scl = (double*)(smem + sb + kOffScratch);
      for (int k = lane; k < EG_N_ACTIONS; k += 32) scl[k] = __ldg(&p.policy->scaled_sorted[y][k]);
      ((uint16_t*)(smem + sb + kOffSortIdx))[lane] = __ldg((const uint16_t*)p.policy->sorted_idx[y] + lane);
      __syncwarp();
    }
  }

  __device__ __forceinline__ void update_deficit_weights(int y, int action, double improvement) {  // deficit.rs:82-135
    const int t = action / 3;
    const int key = deficit_key_of_type(t);
    if (action >= 45 || key == 0xF || action - 3 * t != 0) return;
    const double lr = p.policy->learning_rate;
    const double adj = improvement > 0.0 ? 1.0 + (lr * improvement * 1.5) : ddiv(1.0, 1.0 + (lr * fabs(improvement) * 1.5));
    const double boost = 1.0 + (lr * 0.1);
    double* ldw = LDW(y);
    if (lane < 14) {
      if (lane == key) ldw[lane] = fmin(fmax(ldw[lane] * adj, egrule::kMinWeight), egrule::kMaxWeight);
      else if (improvement < 0.0) ldw[lane] = fmin(ldw[lane] * boost, egrule::kMaxWeight);
    }
    dw_dirty = true;
    __syncwarp();
  }
  __device__ __forceinline__ void update_weights(int y, int action, double improvement) {  // learning.rs:21-88
    const double lr = p.policy->learning_rate;
    const double rel = p.policy->relative_improvement;
    const double immediate = rel > 0.0 ? 0.7 : 0.3;
    const double combined = immediate * improvement + (1.0 - immediate) * rel;
    double* lw = LW(y);
    if (combined == 0.0) {
      // adjustment = 1 / (1 + 0) = 1 and nobody is boosted: the row keeps its values (any weight inside the clamp range,
      // as every weight the rules produce is), and stays clean, so the snapshot's totals and sorted row remain valid.
      // The common case: a plant without CO2 built while emissions are above zero has impact 0 (scoring.rs:60-66).
      const double w0 = lw[action];
      if (w0 >= egrule::kMinWeight && w0 <= egrule::kMaxWeight) return;
    }
    const double adj = combined > 0.0 ? 1.0 + (lr * combined) : ddiv(1.0, 1.0 + (lr * fabs(combined)));
    const double boost = 1.0 + (lr * 0.1);
    for (int k = lane; k < EG_N_ACTIONS; k += 32) {
      if (k == action) lw[k] = fmin(fmax(lw[k] * adj, egrule::kMinWeight), egrule::kMaxWeight);
      else if (combined < 0.0 && k < 45) lw[k] = fmin(lw[k] * boost, egrule::kMaxWeight);
      else if (combined < 0.0 && k == EG_ACT_DO_NOTHING && p.policy->noop_boost) lw[k] = fmin(lw[k] * (1.0 + lr * 0.2), egrule::kMaxWeight);
    }
    rows_dirty = true;
    sorted_valid = false;
    total_valid = false;
    __syncwarp();
  }

  // ---- sampling (canonical key order replaces HashMap iteration order) ---------------------------------------
  __device__ __forceinline__ int sample_deficit_action(int y, uint32_t* replay_pos) {  // sampling.rs:240-378
    if (EG_OPT(p.replay_best)) {
      if (p.policy->has_best && *replay_pos < p.policy->n_best_deficit[y]) return p.policy->best_deficit[p.policy->best_deficit_off[y] + (*replay_pos)++];
      return smart_deficit_fallback_pick(index(93));
    }
    const bool explore = f64() < p.policy->exploration_rate;
    if (explore) return deficit_key_action((int)index(14));
    const double* ldw = LDW(y);
    double total;
    if (dw_dirty) {
      total = 0.0;
      #pragma unroll kScanUnroll
      for (int k = 0; k < 14; k++) total += ldw[k];
    } else {
      total = __ldg(&p.policy->dw_total[y]);  // same left-to-right sum, done once per snapshot on the host
    }
    if (total <= 0.0) return kGasPeaker100;
    double rv = f64() * total;
    #pragma unroll kScanUnroll
    for (int k = 0; k < 14; k++) {
      rv -= ldw[k];
      if (rv <= 0.0) return deficit_key_action(k);
    }
    return kGasPeaker100;
  }
  __device__ __forceinline__ uint32_t sample_additional_actions(int y, uint32_t deficit_count) {  // sampling.rs:380-443
    const uint32_t max_possible = deficit_count >= 20 ? 0 : 20 - deficit_count;
    if (max_possible == 0) return 0;
    const double random_val = f64();
    if (LEAN || p.policy->has_count_weights) {
      const double total = __ldg(&p.policy->cw_total[y]);
      const double* lcw = LCW(y);
      if (total <= 0.0) return 0;
      double rc = random_val * total;
      #pragma unroll kScanUnroll
      for (int c = 0; c < EG_N_COUNT_KEYS; c++) {
        rc -= lcw[c];
        if (rc <= 0.0) return min((uint32_t)c, max_possible);
      }
      return min(5u, max_possible);
    }
    const double scaled_eps = sqrt(p.policy->exploration_rate);  // powf(0.5) of a non-negative value
    const uint32_t min_actions = (uint32_t)round(ddiv(2.0, scaled_eps)), max_actions = (uint32_t)round(ddiv(12.0, scaled_eps));
    const uint32_t cmax = min(max_actions, max_possible), cmin = min(min_actions, cmax);
    if (cmin == cmax) return cmin;
    return cmin + index(cmax - cmin + 1);
  }

  __device__ __forceinline__ int sample_action(int y, uint32_t* replay_pos) {  // sampling.rs:76-238
    if (EG_OPT(p.replay_best)) {
      if (p.policy->has_best && *replay_pos < p.policy->n_best[y]) return p.policy->best[p.policy->best_off[y] + (*replay_pos)++];
      return smart_fallback_pick(y, index(smart_fallback_total(y)));
    }
    const bool explore = f64() < p.policy->action_exploration;  // exploration_rate / (1 + 0.01 iwi) once iwi > 100, per snapshot
    if (explore) return (int)index(EG_N_ACTIONS);
    const double* lw = LW(y);
    double total;
    if (rows_dirty) {
      if (!total_valid) {
        double t = 0.0;
        #pragma unroll kScanUnroll
        for (int k = 0; k < EG_N_ACTIONS; k++) t += lw[k];
        if (lane == 0) VARS()[kVLwTotal] = t;
        total_valid = true;
        __syncwarp();
      }
      total = VARS()[kVLwTotal];
    } else {
      total = __ldg(&p.policy->w_total[y]);
    }
    if (total <= 0.0) return kGasPeaker100;
    if (stagnation()) {
      // stagnation branch (sampling.rs:190-220): weights^power in stable descending order. The sorted row lives in the
      // scratch area: copied from the host-built snapshot row at the start of the year (load_rows), rebuilt on the
      // device after this episode edited the year's weights (sort_local).
      const double* scl = (const double*)(smem + sb + kOffScratch);
      if (rows_dirty && !sorted_valid) {
        sort_local(sb, sb + kOffRows + (uint32_t)(y & 1) * kRowBytes, lane, p.policy->stagnation_power);
        sorted_valid = true;
        double t = 0.0;  // left-to-right sum of the scaled row, once per edit of the row
        #pragma unroll kScanUnroll
        for (int k = 0; k < EG_N_ACTIONS; k++) t += scl[k];
        if (lane == 0) VARS()[kVScaledTotal] = t;
        __syncwarp();
      }
      const double total_scaled = rows_dirty ? VARS()[kVScaledTotal] : __ldg(&p.policy->scaled_total[y]);
      double rv = f64() * total_scaled;
      #pragma unroll kScanUnroll
      for (int k = 0; k < EG_N_ACTIONS; k++) {
        rv -= scl[k];
        if (rv <= 0.0) return (smem + sb + kOffSortIdx)[k];
      }
      return (smem + sb + kOffSortIdx)[0];
    }
    double rv = f64() * total;
    {
      // Decide the scan from a warp-parallel prefix sum when no partial sum comes near
      // the draw. The sequential chain rv_k = fl(rv_{k-1} - w_k) and the tree sums S_k both differ from the exact
      // rv - sum(w_0..w_k) by less than 61 * 2^-52 * total (~1e-14 * total); if every |rv - S_k| exceeds 1e-9 * total, the
      // signs of all rv_k equal the signs of rv - S_k, so the first key with rv_k <= 0 is the first with rv - S_k <= 0.
      // Otherwise (probability ~1e-7 per draw), and when no key crosses, the sequential scan below decides.
      const int k0 = 2 * lane, k1 = 2 * lane + 1;  // lane l holds keys 2l and 2l+1
      const double a = k0 < EG_N_ACTIONS ? lw[k0] : 0.0;
      const double b = k1 < EG_N_ACTIONS ? lw[k1] : 0.0;
      double s = a + b;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const double t = __shfl_up_sync(kFull, s, d);
        if (lane >= d) s += t;
      }
      const double d1 = rv - s, d0 = rv - (s - b);
      const double margin = total * 1e-9;
      const bool near = (k0 < EG_N_ACTIONS && fabs(d0) <= margin) || (k1 < EG_N_ACTIONS && fabs(d1) <= margin);
      const unsigned m0 = __ballot_sync(kFull, k0 < EG_N_ACTIONS && d0 <= 0.0);
      const unsigned m1 = __ballot_sync(kFull, k1 < EG_N_ACTIONS && d1 <= 0.0);
      if (!__any_sync(kFull, near) && (m0 | m1) != 0u) {
        const int f0 = m0 ? 2 * (__ffs((int)m0) - 1) : 1000;
        const int f1 = m1 ? 2 * (__ffs((int)m1) - 1) + 1 : 1000;
        return min(f0, f1);
      }
    }
    #pragma unroll kScanUnroll
    for (int k = 0; k < EG_N_ACTIONS; k++) {
      rv -= lw[k];
      if (rv <= 0.0) return k;
    }
    return kGasPeaker100;
  }

  // record_action / record_deficit_action (simulation.rs:406-409,197): the next slot of the episode's record
  __device__ __forceinline__ void record(int action, int site) {
    if (rec_used >= EG_TRAJ_CAPACITY) { flags |= EG_FLAG_RECORD_OVERFLOW; return; }
    if (lane == 0) {
      if (p.traj) p.traj[ep].actions[rec_used] = (uint8_t)action;
      if (EG_OPT(p.sites)) p.sites[ep].site[rec_used] = site >= 0 ? (uint16_t)site : (uint16_t)EG_SITE_NONE;
    }
    rec_used++;
  }

  __device__ __forceinline__ void run(uint32_t ep_) {
    ep = ep_;
    rec_used = 0;
    uint32_t in_row = 0;  // REPLAY: first slot of the current year's row in the input record
    rng_id = p.same_stream ? 0ull : p.first_episode + ep;
    draw = 0; rbase = 0x80000000u; rbuf = 0ull;
    n_gens = 0; n_offs = 0; flags = 0;
    gcost = 0.0; ocost = 0.0; gen0 = gen1 = gen2 = 0.0; co2 = 0.0;
    __syncwarp();
    const eg_traj* in = REPLAY ? p.replay_in + ep : nullptr;
    uint32_t n_def_total = 0, n_add_total = 0;
    double* vars = VARS();
    const bool learn = !REPLAY && !EG_OPT(p.replay_best);
    if (!REPLAY) prefetch_rows(0);

    for (int y = 0; y < EG_NY; y++) {
      year_start(y);
      bool deficit_mode = ((gen0 + gen1 + gen2) - __ldg(&T->year[y].usage_total)) < 0.0;  // simulation.rs:137
      folded = deficit_mode || EG_OPT(p.yearly != nullptr) || y == EG_NY - 1;
      State cur;                                             // state of the map after the latest change (deficit years)
      cur.net = cur.opinion = cur.cost = 0.0;
      cur.balance = 0.0;
      if (folded) {
        year_folds(y);
        cur = state(y);
      }
      if (!REPLAY) load_rows(y);  // after the folds: both stage data in the scratch area
      if (deficit_mode && lane == 0) {                       // initial state of handle_power_deficit, simulation.rs:341-356
        vars[kVInitNet] = cur.net; vars[kVInitOpinion] = cur.opinion; vars[kVInitBalance] = cur.balance; vars[kVInitCost] = cur.cost;
      }
      double remaining = deficit_mode ? -cur.balance : 0.0;  // Map::handle_power_deficit returns it unchanged (Q2)
      uint32_t attempts = 0, n_def = 0, n_add = 0, n_to_add = 0, replay_def = 0, replay_act = 0;
      bool counted = false;
      // a malformed count never reads past the record: the row is cut at the capacity
      const uint32_t in_def = REPLAY ? min((uint32_t)in->n_deficit[y], (uint32_t)EG_TRAJ_CAPACITY - in_row) : 0;
      const uint32_t in_add = REPLAY ? min((uint32_t)in->n_additional[y], (uint32_t)EG_TRAJ_CAPACITY - in_row - in_def) : 0;
      const uint32_t rec_year = rec_used;  // first slot of this year's row in the record

      for (;;) {
        int action;
        bool is_def;
        if (deficit_mode) {
          if (remaining > 0.0) {                             // simulation.rs:358
            attempts++;
            if (REPLAY) { action = replay_def < in_def ? in->actions[in_row + replay_def] : kBattery100; replay_def++; }
            else action = attempts < 5 ? sample_deficit_action(y, &replay_def) : kBattery100;
            // "Only add a generator if the sampled action is an AddGenerator" (simulation.rs:396-397): anything else is
            // neither applied nor recorded and the loop tries again (recorded trajectories can contain such entries)
            if (action >= 45) continue;
            is_def = true;
          } else {                                           // simulation.rs:490-519
            if (learn) {
              __syncwarp();
              State initial;
              initial.net = vars[kVInitNet]; initial.opinion = vars[kVInitOpinion]; initial.balance = vars[kVInitBalance]; initial.cost = vars[kVInitCost];
              const double overall_success = action_impact(initial, cur);
              if (cur.balance >= 0.0 && overall_success > 0.0 && n_def > 0) {
                const double success_factor = 0.1 * overall_success;
                // this year's deficit actions are the AddGenerator(type, 100 %) keys of the last n_def plants of the list
                if (n_gens >= n_def)
                  for (uint32_t i = 0; i < n_def; i++) update_deficit_weights(y, 3 * (int)(GAT()[n_gens - n_def + i] & 0xF), success_factor);
              }
            }
            deficit_mode = false;
            continue;
          }
        } else if (!counted) {                               // simulation.rs:144-187
          if (REPLAY) n_to_add = in_add;
          else if (EG_OPT(p.replay_best)) n_to_add = p.policy->has_best ? p.policy->n_best[y] : 0;
          else n_to_add = sample_additional_actions(y, n_def);
          counted = true;
          continue;
        } else if (n_add < n_to_add) {                       // simulation.rs:189-198
          if (REPLAY) {
            action = in->actions[in_row + in_def + n_add];
          } else {
            action = sample_action(y, &replay_act);
          }
          is_def = false;
        } else {
          break;
        }

        int site = -1;
        if (action < 45) {                                   // apply_action, actions.rs:42-76
          const int t = action / 3, m = action - 3 * t;
          stash(cur, remaining);
          const int cell = place(t, y);
          unstash(cur, remaining);
          if (cell < 0) flags |= EG_FLAG_NO_SITE;
          else {
            site = (cell >> 8) * p.map.grid_n + (cell & 0xFF);
            if (!add_generator(cell, t, m, y) && is_def) site = -1;  // plant list full: the deficit loop is left like below
          }
        } else if (action < 57) {                            // actions.rs:129-179
          const int a = action - 45;
          const int ot = a / 3;
          add_offset(ot, a - 3 * ot, y);
        }                                                    // 57..60: no generator id matches / DoNothing (Q4)
        // no site with score > 0, or no room for another plant: flagged, the deficit loop is left (it could never end otherwise)
        if (is_def && site < 0) { remaining = 0.0; continue; }
        record(action, site);
        if (is_def) {
          n_def++;
          // state_before of this iteration (simulation.rs:380-395) is the state after the previous change: `cur`
          const State after = state(y);                      // simulation.rs:412-427
          if (learn) {
            const double overall = action_impact(cur, after);
            const double emis = after.net < cur.net ? ddiv(cur.net - after.net, fmax(fabs(cur.net), 1.0)) : 0.0;
            double cost_imp = 0.0;
            if (after.net < 1000.0) {
              const double cost_change = after.cost - cur.cost;
              cost_imp = ddiv(-cost_change, fmax(fabs(cur.cost), 1.0));
            }
            const double op_imp = after.cost < egrule::kMaxCost * 8.0 ? ddiv(after.opinion - cur.opinion, fmax(1.0 - cur.opinion, 0.1)) : 0.0;
            const double combined = overall * 0.7 + emis * 0.15 + cost_imp * 0.1 + op_imp * 0.05;
            __syncwarp();
            update_deficit_weights(y, action, combined);     // simulation.rs:479
            update_weights(y, action, overall * 0.5);        // simulation.rs:482
          }
          remaining = -fmin(after.balance, 0.0);             // simulation.rs:486
          cur = after;
        } else {
          n_add++;
        }
      }
      __syncwarp();

      if (lane == 0) {  // recorded entries of the year: the deficit actions come first, the record may have been cut
        const uint32_t nd_rec = min(n_def, rec_used - rec_year);
        COUNTS()[y] = (uint16_t)nd_rec; COUNTS()[EG_NY + y] = (uint16_t)(rec_used - rec_year - nd_rec);
      }
      n_def_total += n_def; n_add_total += n_add;
      if (REPLAY) in_row += in_def + in_add;

      // calculate_yearly_metrics, analysis/metrics_calculation.rs:32-175 (only the rows somebody asked for; the
      // episode result needs the 2050 row alone, iteration.rs:57-84)
      if (EG_OPT(p.yearly)) {
        const EgYearRow& yr = T->year[y];
        const double usage = __ldg(&yr.usage_total);
        const double generation = gen0 + gen1 + gen2;
        const double balance = generation - usage;
        const double net = co2 - off_amount;
        const double credit = net >= 0.0 ? 0.0 : (-net) * __ldg(&yr.carbon_price);
        const uint32_t active = __ldg(&yr.ex_active) + n_gens;
        const double total_capital = gcost + ocost;
        const double yearly_capital = y == 0 ? total_capital : total_capital - (vars[kVGcostPrev] + vars[kVOcostPrev]);
        const double sales = (p.energy_sales && balance > 0.0) ? (balance * 8.76) * 50000.0 : 0.0;
        const double yearly_total = yearly_capital + 0.0 + 0.0 - credit - (p.energy_sales ? sales : 0.0);
        double total_cost, total_credit, total_sales;
        if (y == 0) { total_cost = yearly_total; total_credit = credit; total_sales = sales; }
        else { total_cost = vars[kVTotalCost] + yearly_total; total_credit = vars[kVTotalCredit] + credit; total_sales = vars[kVTotalSales] + sales; }
        const double opinion = active > 0 ? ddiv(op_sum, (double)active) : 1.0;
        __syncwarp();
        if (lane == 0) {
          vars[kVTotalCost] = total_cost; vars[kVTotalCredit] = total_credit; vars[kVTotalSales] = total_sales;
          eg_year_metrics& m = p.yearly[ep].y[y];
          m.total_population = __ldg(&yr.pop_total);
          m.active_generators = active;
          m.total_power_usage = usage;
          m.total_power_generation = generation;
          m.power_balance = balance;
          m.average_public_opinion = opinion;
          m.yearly_capital_cost = yearly_capital;
          m.total_capital_cost = total_capital;
          m.inflation_factor = __ldg(&yr.inflation);
          m.total_co2_emissions = co2;
          m.total_carbon_offset = off_amount;
          m.net_co2_emissions = net;
          m.yearly_carbon_credit_revenue = credit;
          m.total_carbon_credit_revenue = total_credit;
          m.yearly_energy_sales_revenue = sales;
          m.total_energy_sales_revenue = total_sales;
          m.yearly_total_cost = yearly_total;
          m.total_cost = total_cost;
          m.reserved = 0.0;
        }
        __syncwarp();
      }
    }

    // SimulationMetrics from the 2050 state (iteration.rs:57-84); nothing changed since the last year's actions
    const EgYearRow& last = T->year[EG_NY - 1];
    const double r_net = co2 - off_amount;
    const uint32_t r_active = __ldg(&last.ex_active) + n_gens;
    const double r_opinion = r_active > 0 ? ddiv(op_sum, (double)r_active) : 1.0;
    const double r_cost = gcost + ocost;
    const double r_rel = ((gen0 + gen1 + gen2) - __ldg(&last.usage_total)) >= 0.0 ? 1.0 : 0.0;

    // score_metrics, scoring.rs:5-45 (ln evaluated on the device: <= 1 ulp from the host libm)
    double score;
    {
      const double normalized_cost = fmax(ddiv(r_cost, egrule::kMaxCost), 1.0);
      // ln(1) = 0 whenever the cost is within budget: no logarithm and no zero-numerator division then
      const double cost_term = normalized_cost == 1.0 ? 0.0 : fmin(ddiv(log(normalized_cost), p.ln100), 1.0);
      if (p.cost_only) score = 2.0 - cost_term;
      else if (r_net > 0.0) score = 1.0 - fmin(ddiv(r_net, egrule::kMaxEmissions), 1.0);
      else {
        const double cost_score = 1.0 - cost_term;
        const double cost_weight = normalized_cost > 8.0 ? 0.8 : 0.5;
        const double opinion_weight = 1.0 - cost_weight;
        score = 1.0 + (cost_score * cost_weight + r_opinion * opinion_weight);
      }
    }
    if (lane < 8) {  // eg_result, 64 B: one 8-byte word per lane
      unsigned long long word;
      switch (lane) {
        case 0: word = (unsigned long long)__double_as_longlong(score); break;
        case 1: word = (unsigned long long)__double_as_longlong(r_net); break;
        case 2: word = (unsigned long long)__double_as_longlong(r_opinion); break;
        case 3: word = (unsigned long long)__double_as_longlong(r_cost); break;
        case 4: word = (unsigned long long)__double_as_longlong(r_rel); break;
        case 5: word = (unsigned long long)n_gens | ((unsigned long long)n_offs << 32); break;
        case 6: word = (unsigned long long)(n_def_total & 0xFFFFu) | ((unsigned long long)(n_add_total & 0xFFFFu) << 16) | ((unsigned long long)flags << 32); break;
        default: word = 0ull; break;
      }
      ((unsigned long long*)(p.out + ep))[lane] = word;
    }
    // per-year counts (n_deficit[26] then n_additional[26] are contiguous), then the unused tail of the record: zero
    // actions, EG_SITE_NONE sites (single slots up to the next 8-byte boundary, then words)
    __syncwarp();
    const uint32_t tail8 = (rec_used + 7u) & ~7u;
    if (p.traj) {
      uint8_t* a = p.traj[ep].actions;
      if (lane < EG_NY) ((uint32_t*)p.traj[ep].n_deficit)[lane] = ((const uint32_t*)COUNTS())[lane];
      if (rec_used + lane < tail8) a[rec_used + lane] = 0;
      for (uint32_t i = tail8 / 8 + lane; i < EG_TRAJ_CAPACITY / 8; i += 32) ((unsigned long long*)a)[i] = 0ull;
    }
    if (EG_OPT(p.sites)) {
      uint16_t* st = p.sites[ep].site;
      const uint32_t tail4 = (rec_used + 3u) & ~3u;
      for (uint32_t i = rec_used + lane; i < tail4; i += 32) st[i] = (uint16_t)EG_SITE_NONE;
      for (uint32_t i = tail4 / 4 + lane; i < EG_TRAJ_CAPACITY / 4; i += 32) ((unsigned long long*)st)[i] = ~0ull;
    }
    __syncwarp();
  }
};

// Blocks of 4 warps x 5 per SM, or (medium maps: one larger factor table per block) 10 warps x 2: 20 warps per SM, register cap 96.
// The placement evaluation keeps four table lookups in flight per group of plants and needs ~115 registers to be scheduled that way
// with the episode's state in registers; the state (13 doubles) therefore waits in shared memory while the placement walk runs
// (Warp::stash), which brings the kernel to 94 registers without spills and 20 warps per SM: 3.15 ms per 65,536 episodes against
// 3.39 ms with 4 blocks at 118 registers and 3.55 ms with 5 blocks and no stash (profiles/r02_eval_loop.md).
template <int GEOM> struct Shape {
  static constexpr int kWarps = GEOM == 1 ? 10 : 4, kMinBlocks = GEOM == 1 ? 2 : 5;
};
// kMinBlocks blocks fit in the 227 KB of shared memory of an SM with the largest factor table near_geom admits (the general form
// has none); the system reserves 1 KB per block
static_assert(Shape<0>::kMinBlocks * (Shape<0>::kWarps * kSliceBytes + 8 * EG_COMPACT_MAX_FACTORS + 1024) <= 227 * 1024, "compact maps");
static_assert(Shape<1>::kMinBlocks * (Shape<1>::kWarps * kSliceBytes + 8 * EG_MEDIUM_MAX_FACTORS + 1024) <= 227 * 1024, "medium maps");

template <bool REPLAY, int GEOM, int MODE>
__global__ void __launch_bounds__(32 * Shape<GEOM>::kWarps, Shape<GEOM>::kMinBlocks) eg_episode_kernel(const __grid_constant__ EgEpisodeParams p, int slice_bytes, int table_bytes) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (GEOM != 2) {  // block-shared copy of the distance/radius factors at the start of the shared memory
    double* nf_s = (double*)smem;  // compact: class rc holds its r2_limit[rc] entries from offset r2_limit[6 + rc], then a 1.0
    for (int rc = 0; rc < EG_N_RCLASS; rc++) {
      const int cnt = __ldg(&p.map.r2_limit[rc]), off = __ldg(&p.map.r2_limit[EG_N_RCLASS + rc]);
      for (int i = threadIdx.x; i < cnt + 1; i += blockDim.x)
        nf_s[off + i] = i < cnt ? __ldg(&p.map.near_factor[rc * p.map.r2_stride + i]) : 1.0;
    }
    __syncthreads();
  }
  Warp<REPLAY, GEOM, MODE> w(p, opaque((uint32_t)(table_bytes + warp * slice_bytes)), lane);
  // persistent warps: every warp fetches the next unclaimed episode of the batch until none is left, so a short
  // episode never leaves its warp idle while the block's longest one finishes
  for (;;) {
    uint32_t ep = 0;
    if (lane == 0) ep = atomicAdd(p.next_episode, 1u);
    ep = __shfl_sync(kFull, ep, 0);
    if (ep >= p.n) break;
    w.run(ep);
  }
}

template <bool REPLAY, int GEOM, int MODE>
cudaError_t launch_as(const EgEpisodeParams& p, cudaStream_t stream) {
  constexpr int warps = Shape<GEOM>::kWarps;
  const int shared_tab = GEOM == 2 ? 0 : (p.nf_entries * (int)sizeof(double) + 15) & ~15;
  const size_t smem_bytes = (size_t)warps * kSliceBytes + shared_tab;
  if (smem_bytes > 227 * 1024) return cudaErrorInvalidConfiguration;
  // function attributes and the occupancy query are per (device, shared-memory size): done once, then cached
  struct Cached { size_t smem = 0; int resident = 0; };
  static thread_local Cached cache[64];
  int dev = 0;
  cudaError_t err = cudaGetDevice(&dev);
  if (err != cudaSuccess) return err;
  Cached local;
  Cached& shape = (dev >= 0 && dev < 64) ? cache[dev] : local;
  if (shape.smem != smem_bytes || shape.resident == 0) {
    err = cudaFuncSetAttribute(eg_episode_kernel<REPLAY, GEOM, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (err != cudaSuccess) return err;
    // shared-memory carveout: room for the kMinBlocks blocks the register budget allows, the rest stays L1
    const int carveout = std::min(100, (int)((Shape<GEOM>::kMinBlocks * (smem_bytes + 1024) * 100 + 228 * 1024 - 1) / (228 * 1024)));
    cudaFuncSetAttribute(eg_episode_kernel<REPLAY, GEOM, MODE>, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
    // grid = every block the device can hold at once (a multiple of the SM count), never more warps than episodes
    int sms = 0, per_sm = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eg_episode_kernel<REPLAY, GEOM, MODE>, 32 * warps, smem_bytes);
    if (err != cudaSuccess) return err;
    if (per_sm < 1) return cudaErrorInvalidConfiguration;
    shape.smem = smem_bytes;
    shape.resident = sms * per_sm;
  }
  uint32_t blocks = std::min<uint32_t>((uint32_t)shape.resident, (p.n + warps - 1) / warps);
  if (blocks == 0) return cudaErrorInvalidConfiguration;
  err = cudaMemsetAsync(p.next_episode, 0, sizeof(uint32_t), stream);
  if (err != cudaSuccess) return err;
  eg_episode_kernel<REPLAY, GEOM, MODE><<<blocks, 32 * warps, smem_bytes, stream>>>(p, kSliceBytes, shared_tab);
  return cudaGetLastError();
}

template <bool REPLAY>
cudaError_t launch(const EgEpisodeParams& p, cudaStream_t stream) {
  if (p.n == 0) return cudaSuccess;
  // the training launch (no per-year or per-site outputs, sampling from the weights, count weights present) runs a lean
  // instantiation without the code of those options: the kernel is bound by instruction fetch, and 8 KB of code that
  // never executes still spreads the hot instructions over more cache lines (-10 % time on trained tables)
  const int geom = p.map.near_geom;
  if (!REPLAY && !p.yearly && !p.sites && !p.replay_best && p.count_weights) {
    if (p.stagnation) return geom == 0 ? launch_as<false, 0, 2>(p, stream) : geom == 1 ? launch_as<false, 1, 2>(p, stream) : launch_as<false, 2, 2>(p, stream);
    return geom == 0 ? launch_as<false, 0, 1>(p, stream) : geom == 1 ? launch_as<false, 1, 1>(p, stream) : launch_as<false, 2, 1>(p, stream);
  }
  return geom == 0 ? launch_as<REPLAY, 0, 0>(p, stream) : geom == 1 ? launch_as<REPLAY, 1, 0>(p, stream) : launch_as<REPLAY, 2, 0>(p, stream);
}

}  // namespace

cudaError_t eg_launch_rollout(const EgEpisodeParams& p, cudaStream_t stream) { return launch<false>(p, stream); }
cudaError_t eg_launch_replay(const EgEpisodeParams& p, cudaStream_t stream) { return launch<true>(p, stream); }
