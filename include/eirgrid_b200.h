/*
 * eirgrid_b200.h — C ABI of the B200-native episode-rollout engine for GridAI (ETM-Code/eirgrid).
 *
 * The reference has no FFI layer; the seam this library sits behind is the body of the rayon
 * `into_par_iter` closure in aiSimulator/src/core/multi_simulation.rs:427-610:
 *
 *     run_iteration(i, &mut map, &mut local_weights, replay_best, seed, ...)   core/iteration.rs:10-20
 *     weights.transfer_recorded_actions_from / apply_contrast_learning /
 *     update_best_strategy / apply_deficit_contrast_learning                   multi_simulation.rs:494-508
 *     ActionWeights::{new, load_from_file, save_to_file, update_weights_from}  ai/learning/weights/ (all .rs)
 *     load_settlements / load_generators / coastline_points.json               data/ (loaders), map_handler.rs:360-375
 *
 * Every entry point below names the reference interface it replaces. All pointers are plain
 * host or device pointers (stated per function); no C++/torch types cross this boundary.
 * Functions return 0 on success or a negative eg_status; eg_last_error() gives the message.
 * A context is thread-compatible (one call in flight per ctx), one context per GPU/process.
 */
#ifndef EIRGRID_B200_H
#define EIRGRID_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- fixed sizes of the path (config/constants.rs, ai/learning/constants.rs) ---------------- */
#define EG_BASE_YEAR 2025              /* constants.rs:2 */
#define EG_END_YEAR 2050               /* constants.rs:3 */
#define EG_N_YEARS 26
#define EG_N_GEN_TYPES 15              /* models/generator.rs:11-36, enum order */
#define EG_N_OFFSET_TYPES 4            /* insertion order of weights/core.rs:100-114: Forest, Wetland, ActiveCapture, CarbonCredit */
#define EG_N_MULTS 3                   /* cost multipliers 100/120/150 %, constants.rs:333-335 */
#define EG_N_ACTIONS 61                /* regular action keys per year, weights/core.rs:35-120 */
#define EG_N_DEFICIT_KEYS 15           /* weights/core.rs:130-152 */
#define EG_N_COUNT_KEYS 21             /* action counts 0..=20, weights/core.rs:163 */
#define EG_TRAJ_CAPACITY 984           /* action slots per EPISODE in eg_traj; year rows are stored back to back (CSR), so a
                                          single year may hold all of them. The reference's Vec<GridAction> lists are unbounded
                                          (simulation.rs:406-409, strategy.rs:188-196); an episode that outgrows the capacity is
                                          flagged EG_FLAG_RECORD_OVERFLOW. Training episodes stay below 26 x ~21 actions; the
                                          plant capacity (EG_MAX_NEW_GENERATORS) is reached first in compounding replay runs. */
#define EG_BEST_CAPACITY (2 * EG_TRAJ_CAPACITY)  /* best_actions of a replay iteration hold every additional action twice (quirk Q10) */
#define EG_SITE_NONE 0xFFFFu

/* Action codes (uint8) — canonical key order == insertion order in ActionWeights::new:
 *   0..44  AddGenerator(type t, mult m)      code = 3*t + m        (m: 0=100 %, 1=120 %, 2=150 %)
 *   45..56 AddCarbonOffset(type o, mult m)   code = 45 + 3*o + m
 *   57 UpgradeEfficiency("")  58 AdjustOperation("",0)  59 CloseGenerator("")  60 DoNothing
 * Deficit key k (0..14) maps to an action code through eg_deficit_key_action(k). */
#define EG_ACT_UPGRADE 57
#define EG_ACT_ADJUST 58
#define EG_ACT_CLOSE 59
#define EG_ACT_DO_NOTHING 60

typedef enum {
  EG_OK = 0,
  EG_ERR_INVALID = -1,      /* bad argument */
  EG_ERR_IO = -2,           /* file missing / unparsable (reference: Err from the loaders) */
  EG_ERR_CUDA = -3,         /* CUDA runtime error; message carries cudaGetErrorString */
  EG_ERR_NO_DEVICE = -4,    /* no CUDA device: there is NO CPU fallback */
  EG_ERR_STATE = -5,        /* call order (e.g. rollout before a map is loaded) */
  EG_ERR_OVERFLOW = -6      /* an episode exceeded a fixed capacity (reported per episode in flags too) */
} eg_status;

/* eg_result.flags */
#define EG_FLAG_GEN_OVERFLOW 1u     /* more than EG_MAX_NEW_GENERATORS new plants */
#define EG_FLAG_OFFSET_OVERFLOW 2u  /* more than EG_MAX_OFFSETS offsets */
#define EG_FLAG_RECORD_OVERFLOW 4u  /* more than EG_TRAJ_CAPACITY actions in the episode: the simulation applied them all, the record is cut */
#define EG_FLAG_NO_SITE 8u          /* placement search found no site with score > 0 (reference falls back; we flag) */
#define EG_MAX_NEW_GENERATORS 560
#define EG_MAX_OFFSETS 520

typedef struct eg_ctx eg_ctx;         /* device context: stream, static map tables in HBM */
typedef struct eg_weights eg_weights; /* host object == reference ActionWeights (weights/mod.rs:49-107) */

/* ---- per-episode outputs --------------------------------------------------------------------- */
/* SimulationMetrics (ai/metrics/simulation_metrics.rs:5-10) + score_metrics (scoring.rs:5-45). 64 B. */
typedef struct {
  double score;             /* score_metrics(metrics, optimization_mode) */
  double net_emissions;     /* final_net_emissions = 2050 net_co2_emissions        iteration.rs:70 */
  double public_opinion;    /* average_public_opinion of 2050                      iteration.rs:71 */
  double total_cost;        /* 2050 total_capital_cost (quirk Q7)                  iteration.rs:72 */
  double power_reliability; /* 1.0 if 2050 power_balance >= 0 else 0.0             iteration.rs:73 */
  uint32_t n_generators;    /* new plants built in the episode */
  uint32_t n_offsets;
  uint16_t n_deficit_actions;
  uint16_t n_additional_actions;
  uint32_t flags;
  uint32_t reserved;
} eg_result;

/* Recorded actions of one episode. Year y's row is current_deficit_actions[y] followed by the additional actions of
 * year y (== current_run_actions[y], simulation.rs:406-409,197); the rows of 2025..2050 follow each other without gaps:
 * row y starts at slot sum_{y' < y} (n_deficit[y'] + n_additional[y']). Unused slots are zero. 1088 B. */
typedef struct {
  uint16_t n_deficit[EG_N_YEARS];
  uint16_t n_additional[EG_N_YEARS];
  uint8_t actions[EG_TRAJ_CAPACITY];
} eg_traj;

/* Candidate-site index (i*grid_n + j of find_suitable_location's scan, metal_location_search.rs:120-124)
 * chosen for the action in the same slot of eg_traj; EG_SITE_NONE for actions that place nothing and for unused slots. */
typedef struct {
  uint16_t site[EG_TRAJ_CAPACITY];
} eg_sites;

/* Numeric fields of YearlyMetrics (analysis/metrics.rs:6-31). 144 B. */
typedef struct {
  uint32_t total_population;
  uint32_t active_generators;
  double total_power_usage;
  double total_power_generation;
  double power_balance;
  double average_public_opinion;
  double yearly_capital_cost;
  double total_capital_cost;
  double inflation_factor;
  double total_co2_emissions;
  double total_carbon_offset;
  double net_co2_emissions;
  double yearly_carbon_credit_revenue;
  double total_carbon_credit_revenue;
  double yearly_energy_sales_revenue;
  double total_energy_sales_revenue;
  double yearly_total_cost;
  double total_cost;
  double reserved;
} eg_year_metrics;

typedef struct {
  eg_year_metrics y[EG_N_YEARS];
} eg_yearly;

/* ---- run configuration (mirrors the CLI flags that reach run_iteration, cli/cli.rs:3-59) ------ */
typedef struct {
  uint32_t cost_only;                 /* --cost-only → optimization_mode Some("cost_only") for the driver-side score */
  uint32_t enable_energy_sales;       /* default 1 */
  uint32_t enable_construction_delays;/* default 0; 1 → EG_ERR_INVALID: the reference's deficit loop does not terminate with delays on (DESIGN.md §9) */
  uint32_t replay_best;               /* run_iteration's replay_best_strategy: force_best_actions */
  uint32_t same_stream_all_episodes;  /* quirk Q8 (--seed re-seeds every episode identically); 0 = one stream per episode id */
  uint32_t reserved[3];
} eg_run_cfg;

/* ---- map description for eg_map_set (synthetic maps, config 4) -------------------------------- */
typedef struct {
  uint32_t n_settlements;
  const double* settlement_x;        /* grid metres, already transformed+clamped */
  const double* settlement_y;
  const uint32_t* settlement_pop;    /* 2025 population */
  uint32_t n_existing;
  const double* existing_x;
  const double* existing_y;
  const uint8_t* existing_type;      /* generator type index */
  const double* existing_capacity_mw;
  uint32_t n_coast;
  const double* coast_x;
  const double* coast_y;
  uint32_t grid_n;                   /* distinct candidate sites per axis (reference: 51) */
  double grid_step;                  /* metres between candidate sites (reference: 1000), must be integer-valued */
} eg_map_desc;

/* ---- dense view of the policy table (ActionWeights, weights/mod.rs:49-107) --------------------- */
typedef struct {
  double weights[EG_N_YEARS][EG_N_ACTIONS];
  double deficit_weights[EG_N_YEARS][EG_N_DEFICIT_KEYS];
  double count_weights[EG_N_YEARS][EG_N_COUNT_KEYS];
  double learning_rate;
  double exploration_rate;
  double best_metrics[4];             /* net_emissions, public_opinion, total_cost, power_reliability */
  uint32_t has_count_weights;         /* 0 after load_from_file (weights/serialization.rs:474) */
  uint32_t has_best;
  uint32_t iteration_count;
  uint32_t iterations_without_improvement;
} eg_weights_table;

typedef struct {
  uint32_t n_episodes;
  uint32_t n_improvements;            /* times update_best_strategy replaced the best */
  uint32_t n_contrast_applied;        /* episodes whose deterioration passed the dynamic threshold */
  uint32_t iterations_without_improvement;
  double best_score;
  double batch_best_score;
  int64_t batch_best_episode;         /* index inside the batch, -1 if none */
  uint32_t n_flagged;                 /* episodes of the batch with eg_result.flags != 0 (capacity overflow, no site found) */
  uint32_t reserved;
} eg_update_stats;

/* ---- context ----------------------------------------------------------------------------------- */
/* One context per process/GPU. `cuda_stream` may be NULL (own stream) or a cudaStream_t the caller
 * owns (e.g. torch.cuda.current_stream().cuda_stream) so that CUDA events recorded by the caller see
 * the kernels. Fails with EG_ERR_NO_DEVICE when no GPU is present. */
int eg_init(int device, void* cuda_stream, eg_ctx** out);
void eg_destroy(eg_ctx* ctx);
const char* eg_last_error(void);
int eg_sync(eg_ctx* ctx);
/* number of kernel launches issued by this library since eg_init (for bench.py's gpu_launches) */
uint64_t eg_kernel_launches(const eg_ctx* ctx);

/* ---- map loading: replaces load_settlements (settlements_loader.rs:23-42), load_generators
 * (generators_loader.rs:133-207), the coastline include (map_handler.rs:360-375) and
 * initialize_map (main.rs:74-193). Builds the static site tables on the GPU (replaces
 * MetalLocationSearch's per-call scan, gpu/metal_location_search.rs:110-176). ---------------------- */
int eg_map_load(eg_ctx* ctx, const char* settlements_json, const char* generators_csv, const char* coastline_json);
int eg_map_set(eg_ctx* ctx, const eg_map_desc* desc);
/* sizes of the loaded map: n_settlements, n_existing, n_coast, grid_n */
int eg_map_info(const eg_ctx* ctx, uint32_t out[4]);
/* copy back static site tables for inspection/tests: prefix score after settlements+existing plants for
 * radius class `rclass` (0..5) in `year`, and final static score/order for placement class `pclass` (0..6).
 * Any pointer may be NULL. Host buffers of n_sites entries. */
int eg_map_site_tables(eg_ctx* ctx, uint32_t year_index, uint32_t rclass, uint32_t pclass,
                       double* prefix_score, double* static_score_sorted, uint32_t* order_sorted);

/* per-site static factors: 1/(1+min_coast_distance/5000) and the average settlement opinion of a plant on the site */
int eg_map_site_static(eg_ctx* ctx, double* coast_factor, double* site_opinion);

/* ---- policy table: replaces ActionWeights::new (weights/core.rs:25-250), load_from_file /
 * save_to_file (weights/serialization.rs:29-493), update_weights_from (strategy.rs:281-311) ------- */
int eg_weights_new(eg_weights** out);
void eg_weights_free(eg_weights* w);
int eg_weights_clone(const eg_weights* src, eg_weights** out);
int eg_weights_load_json(const char* path, eg_weights** out);
int eg_weights_save_json(const eg_weights* w, const char* path);
int eg_weights_merge(eg_weights* dst, const eg_weights* other);
/* --track-weight-history: append one snapshot {iteration, timestamp (RFC 3339), weights: ActionWeights::to_json(), best_score}
 * to the JSON array in `history_path` (created if missing) — save_weight_history, core/multi_simulation.rs:179-207, with
 * to_json of weights/serialization.rs:495-540: the file aiSimulator/tools/visualization/weight_history_animation.py reads. */
int eg_weights_history_append(const eg_weights* w, uint64_t iteration, const char* history_path);
int eg_weights_get_table(const eg_weights* w, eg_weights_table* out);
int eg_weights_set_table(eg_weights* w, const eg_weights_table* in);
/* best strategy lists (best_actions / best_deficit_actions, Option<HashMap<u32, Vec<GridAction>>>), any length:
 * n_best[y] = len(best_actions[y]) (which already contains the year's deficit actions first, Appendix C of SURVEY.md),
 * n_best_deficit[y] = len(best_deficit_actions[y]); the lists themselves are written back to back, year after year, into
 * `best` / `best_deficit` as far as their capacities reach (either may be NULL to query the lengths only).
 * Returns 1 if a best strategy exists, 0 if not. */
int eg_weights_get_best(const eg_weights* w, uint32_t n_best[EG_N_YEARS], uint8_t* best, size_t best_capacity,
                        uint32_t n_best_deficit[EG_N_YEARS], uint8_t* best_deficit, size_t best_deficit_capacity);
uint8_t eg_deficit_key_action(uint32_t deficit_key);

/* ---- the hot path ------------------------------------------------------------------------------- */
/* Replaces run_iteration → run_simulation (core/iteration.rs:10-95, core/simulation.rs:22-522) for
 * `n` episodes with ids first_episode..first_episode+n-1 sampled from the weights snapshot `w`
 * (== local_weights = shared.read().clone(), multi_simulation.rs:457-460).
 * HOST buffers (pinned recommended); copies are done inside the call on the ctx stream and the call
 * returns after the results are on the host. Any of traj/sites/yearly may be NULL. */
int eg_rollout_batch(eg_ctx* ctx, const eg_weights* w, const eg_run_cfg* cfg, uint64_t seed,
                     uint64_t first_episode, uint32_t n, eg_result* out, eg_traj* traj_out,
                     eg_sites* sites_out, eg_yearly* yearly_out);
/* Same with DEVICE output buffers, asynchronous on the ctx stream (inputs resident: the weights
 * snapshot is uploaded by eg_weights_upload). A call with d_sites == d_yearly == NULL, replay_best == 0 and a snapshot
 * that has count weights (every ActionWeights::new / reference checkpoint has) runs the lean instantiation of the
 * kernel, 10-30 % faster than the general one; results are identical either way. */
int eg_weights_upload(eg_ctx* ctx, const eg_weights* w);
int eg_rollout_batch_device(eg_ctx* ctx, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode,
                            uint32_t n, eg_result* d_out, eg_traj* d_traj, eg_sites* d_sites, eg_yearly* d_yearly);

/* Trajectory replay (BASELINE config 2): re-simulate recorded per-year action lists, no sampling.
 * Replaces run_simulation with the sampling calls (sample_deficit_action / sample_additional_actions /
 * sample_action, sampling.rs:76-443) substituted by reads from `in`. HOST buffers. */
int eg_replay_batch(eg_ctx* ctx, const eg_run_cfg* cfg, const eg_traj* in, uint32_t n, eg_result* out,
                    eg_sites* sites_out, eg_yearly* yearly_out);
int eg_replay_batch_device(eg_ctx* ctx, const eg_run_cfg* cfg, const eg_traj* d_in, uint32_t n,
                           eg_result* d_out, eg_sites* d_sites, eg_yearly* d_yearly);

/* ---- weight update: replaces the write-lock section multi_simulation.rs:494-508
 * (transfer_recorded_actions_from → apply_contrast_learning → update_best_strategy →
 *  apply_deficit_contrast_learning; learning.rs:131-373, strategy.rs:19-258,313-342), applied for the
 * n episodes of a batch in episode-index order. HOST buffers. `replay_best` = the batch ran with
 * eg_run_cfg.replay_best (its doubled action records are rebuilt, quirk Q10); `rng_seed` feeds the randomisation
 * branch (iterations_without_improvement > 1200). */
int eg_update(eg_weights* w, const eg_result* results, const eg_traj* trajs, uint32_t n,
              uint32_t replay_best, uint64_t rng_seed, eg_update_stats* stats_out);

/* The same rule with DEVICE buffers, applied on the GPU in episode-index order (update.cu): `w` ends with the same table,
 * best strategy, counters and improvement history as after eg_update on the same records, bit for bit — both forms take
 * their thresholds and factors from one source (csrc/update_rule.hpp) — at ~20-40 ns per episode instead of 4-11 us. The
 * rule stays sequential in the episodes; the device form finds the running best with a scan over the scores, derives each
 * episode's factors and multiplication counts in parallel and walks the table once, one thread per table entry.
 * Synchronous: returns after `w` has been updated. */
int eg_update_device(eg_ctx* ctx, eg_weights* w, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n,
                     uint32_t replay_best, uint64_t rng_seed, eg_update_stats* stats_out);
/* One batch of the reference's loop on one GPU (the par_iter closure for n episodes that share one snapshot,
 * multi_simulation.rs:457-508): snapshot H2D, rollout of episodes first_episode..+n, in-order update on the device, state
 * D2H. Episode results stay on the device: eg_train_batch_results copies them out. */
int eg_train_batch_inorder(eg_ctx* ctx, eg_weights* w, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode, uint32_t n,
                           uint64_t rng_seed, eg_update_stats* stats_out);

/* Batch-synchronous update for sharded episodes (DESIGN.md §update): eg_update_stats_device accumulates a rank's
 * statistics on the device into a table of EG_STATS_WORDS int64 words and finds the rank's best episode, and
 * eg_update_pack_best_device packs that episode as the rank's winner record. The ranks all-gather
 * [statistics table | winner record]; every rank then calls eg_update_combine_apply, which sums the tables, picks the batch
 * winner among the records and applies the identical update (eg_update_apply_stats). */
#define EG_STATS_WORDS (8 + EG_N_YEARS * (3 * EG_N_ACTIONS + EG_N_DEFICIT_KEYS))
int eg_update_stats_device(eg_ctx* ctx, const eg_weights* w, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n,
                           int64_t* d_stats /* EG_STATS_WORDS, accumulated (not cleared) */,
                           double* d_best_score /* [1] max score of the shard */,
                           unsigned long long* d_best_index /* [1] lowest index with that score */);
/* Zero the statistics table on the ctx stream (start of a batch). */
int eg_update_stats_clear_device(eg_ctx* ctx, int64_t* d_stats);
/* This rank's candidate for the batch winner as one flat record on the device, ready for the all-gather:
 * [best score f64 | global episode id i64 | eg_result | eg_traj] (EG_BEST_RECORD_BYTES). d_best_score / d_best_index are
 * the outputs of eg_update_stats_device; global id = first_global_episode + index. d_record is 8-byte aligned. */
#define EG_BEST_RECORD_BYTES (16 + sizeof(eg_result) + sizeof(eg_traj))
int eg_update_pack_best_device(eg_ctx* ctx, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n,
                               const double* d_best_score, const unsigned long long* d_best_index,
                               uint64_t first_global_episode, void* d_record);
int eg_update_apply_stats(eg_weights* w, const int64_t* stats, uint64_t n_total,
                          const eg_result* batch_best_result, const eg_traj* batch_best_traj,
                          int64_t batch_best_index, eg_update_stats* stats_out);

/* One training batch on one GPU, everything on the ctx stream (replaces the par_iter closure for a shard of the batch):
 * weights snapshot H2D, rollout of episodes first_episode..+n, update statistics, the shard's winner record, both
 * copied to pinned host memory. _begin returns once the work is queued (several contexts/GPUs can run concurrently from
 * one host thread); _end waits and copies out the EG_STATS_WORDS int64 statistics (this shard only) and the
 * EG_BEST_RECORD_BYTES winner record. Episode results stay on the device: eg_train_batch_results copies them out. */
int eg_train_batch_begin(eg_ctx* ctx, const eg_weights* w, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode, uint32_t n);
int eg_train_batch_end(eg_ctx* ctx, int64_t* stats_out, void* record_out);
int eg_train_batch_results(eg_ctx* ctx, eg_result* out, eg_traj* traj_out /* nullable */);
/* Host side of the exchange step, identical on every rank/GPU: `stats_sum` = element-wise sum of the shards' statistics,
 * `records` = n_records winner records back to back; the winner is the highest score, lowest global episode id among
 * equals; then eg_update_apply_stats. first_episode = global id of the batch's first episode. */
int eg_update_combine_apply(eg_weights* w, const int64_t* stats_sum, const void* records, uint32_t n_records,
                            uint64_t n_total, uint64_t first_episode, eg_update_stats* stats_out);

/* ---- policy evaluation: statistics of n episodes sampled from one table, reduced on the device -------------------------
 * A fixed-size record; the all-zero record is the empty statistics. Moments are {mean, m2 = sum of squared deviations, min,
 * max}, folded with Welford's update inside a block and merged with Chan et al.'s pairwise formula everywhere else. For fixed
 * (weights, cfg, seed, first_episode, n) the record is the same bytes on every run. Integer parts, min/max and the best/worst ids
 * do not depend on how the episode range is split; the moments of a split range differ from the unsplit ones in the last bits. */
#define EG_EVAL_CHUNK 65536            /* episodes rolled out and reduced per step of eg_evaluate */
#define EG_EVAL_SCORE_BINS 2048        /* score histogram over [0, 2]: bin = min(floor(score * 1024), 2047) */
#define EG_EVAL_N_FLAGS 4              /* one counter per EG_FLAG_* bit */
#define EG_EVAL_N_FINAL 9              /* score, net_emissions, public_opinion, total_cost, power_reliability, n_generators, n_offsets,
                                          n_deficit_actions, n_additional_actions (the fields of eg_result in order) */
#define EG_EVAL_N_YEAR_FIELDS 18       /* total_population, active_generators and the 16 f64 fields of eg_year_metrics before `reserved` */
#define EG_EVAL_COUNTER_WORDS (1 + EG_EVAL_N_FLAGS + EG_EVAL_SCORE_BINS + 1 + 3 * EG_N_YEARS + 1 + 2 * EG_N_YEARS * EG_N_ACTIONS)

typedef struct {
  double mean, m2, min, max;
} eg_moments;

typedef struct {
  uint64_t n_episodes;
  uint64_t best_episode;               /* global episode id of the highest score, the lowest id among equal scores (0 if empty) */
  uint64_t worst_episode;              /* the same for the lowest score */
  uint32_t has_yearly;                 /* the per-year moments and counts below are filled */
  uint32_t reserved;
  eg_moments final_metrics[EG_EVAL_N_FINAL];
  eg_moments yearly[EG_N_YEARS][EG_EVAL_N_YEAR_FIELDS];   /* follows final_metrics without a gap */
  /* counters (EG_EVAL_COUNTER_WORDS words from n_flagged to the end): merged by addition */
  uint64_t n_flagged;                  /* episodes with eg_result.flags != 0 */
  uint64_t flag_counts[EG_EVAL_N_FLAGS];
  uint64_t score_hist[EG_EVAL_SCORE_BINS];
  uint64_t score_out_of_range;         /* scores outside [0, 2] and NaN */
  uint64_t net_zero_or_below[EG_N_YEARS];       /* episodes with net_co2_emissions <= 0 in the year (yearly only) */
  uint64_t in_deficit[EG_N_YEARS];              /* episodes with power_balance < 0 in the year (yearly only) */
  uint64_t first_net_zero_year[EG_N_YEARS + 1]; /* first year with net_co2_emissions <= 0; [EG_N_YEARS] = never (yearly only) */
  uint64_t additional_actions[EG_N_YEARS][EG_N_ACTIONS];  /* additional actions by year and code, as stored in eg_traj */
  uint64_t deficit_actions[EG_N_YEARS][EG_N_ACTIONS];     /* deficit-handler actions by year and code */
} eg_eval_stats;

/* n episodes with ids first_episode .. first_episode + n - 1 sampled from w (uploads w as the ctx's snapshot, like
 * eg_rollout_batch), rolled out and reduced on the device in chunks of EG_EVAL_CHUNK episodes; one copy to the host at the
 * end. with_yearly = 0 reduces results and action records only, which runs the lean instantiation of the episode kernel
 * whenever the snapshot allows it; 1 adds the per-year part. n = 0 gives the empty record. */
int eg_evaluate(eg_ctx* ctx, const eg_weights* w, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode, uint64_t n,
                uint32_t with_yearly, eg_eval_stats* out);
/* Folds n episodes already on the device (global ids first_global_episode..) into the DEVICE record *d_acc, asynchronously on
 * the ctx stream, in the chunks eg_evaluate uses. d_yearly may be NULL; every call on one record passes it or none does. */
int eg_eval_accumulate_device(eg_ctx* ctx, const eg_result* d_results, const eg_traj* d_traj, const eg_yearly* d_yearly,
                              uint32_t n, uint64_t first_global_episode, eg_eval_stats* d_acc);
/* Host only, needs no device: dst <- dst followed by src (the shards of an evaluation in episode order). The same merge as
 * the device's, so the bits agree. EG_ERR_INVALID when both are non-empty and only one has the per-year part. */
int eg_eval_stats_merge(eg_eval_stats* dst, const eg_eval_stats* src);
/* The record as JSON (DESIGN.md §4.6): moments as mean / std / min / max, score quantiles from the histogram, per-year
 * moments and probabilities, action counts by name. Host only. */
int eg_eval_stats_write_json(const eg_eval_stats* s, const char* path);

/* ---- CSV export of the best run (SURVEY.md §8(f) N2; utils/csv_export.rs:114-432,456-530 and the call site
 * core/multi_simulation.rs:852-925). The best strategy stored in `w` is replayed on the GPU (eg_replay_batch) and written as
 *   <output_dir>/<%Y%m%d_%H%M%S>/simulation_summary.csv     final metrics, actions taken with estimated costs, yearly summary
 *   <output_dir>/<%Y%m%d_%H%M%S>/improvement_history.csv    the weights' improvement history
 *   <output_dir>/<%Y%m%d_%H%M%S>/yearly_details/settlements.csv
 *   <output_dir>/<%Y%m%d_%H%M%S>/yearly_details/generators.csv       csv_export.rs:532-984: one row per active plant and year
 *   <output_dir>/<%Y%m%d_%H%M%S>/yearly_details/carbon_offsets.csv   csv_export.rs:987-1093
 *   <output_dir>/<%Y%m%d_%H%M%S>/operation_logs/generator_operation_logs.csv   csv_export.rs:1096-1310 (header only, as there)
 * in the reference's column order and number formats, including what its exporter actually does with them: plant rows are
 * rebuilt from the ids with per-type default figures and id-hash coordinates, offsets are still `Planned` on the export
 * map so their offset columns are 0 (DESIGN.md §9 N2 lists these). Row order inside a year (HashMap order in the reference)
 * is plant order; offset coordinates (thread_rng there) come from a fixed Philox stream.
 * `written_dir` (nullable, >= 512 bytes) receives the directory. Returns EG_ERR_STATE if `w` has no best strategy. */
int eg_export_best_run_csv(eg_ctx* ctx, const eg_weights* w, const eg_run_cfg* cfg, const char* output_dir, char* written_dir);

/* ---- location suitability analysis (BASELINE config 5): replaces Map::analyze_locations →
 * LocationAnalysis::analyze_map (map_handler.rs:61-142) and calculate_generator_suitability
 * (map_handler.rs:1319-1396) / the unused MSL kernel computeSuitability (metal:239-258).
 * scores: HOST buffer of n_points*15 doubles, point p = (i+half)*(2*half+1) + (j+half) for
 * i,j in [-half, half] at step 2000 m (negatives clamp to 0 exactly like Coordinate::new).
 * use_loaded_map = 0 reproduces the shipped cache (empty map), 1 uses the loaded settlements/plants. */
int eg_location_analysis(eg_ctx* ctx, int use_loaded_map, int32_t half_steps, double step,
                         double* scores_out, uint32_t first_point, uint32_t n_points);
/* The same with the settlement populations of simulated year 2025 + year_index (they grow 1 % a year and decide the urban
 * test and the nearby-population rule): BASELINE configs[4] asks for all sites x 15 types x 26 years. year_index 0 == above. */
int eg_location_analysis_year(eg_ctx* ctx, int use_loaded_map, uint32_t year_index, int32_t half_steps, double step,
                              double* scores_out, uint32_t first_point, uint32_t n_points);

/* BASELINE configs[4]: every candidate generator site x 15 types x simulated years in ONE pass. Sites are the points
 * (i * step, j * step) for i, j in [0, sites_per_axis) (clamped to the 50 km map like Coordinate::new), site = i * sites_per_axis + j:
 * the placement search's candidate grid is sites_per_axis = 51, step = 1000 (metal_location_search.rs:120-124 after the clamp). A
 * site's geometry (water / near-water / coastal tests, distance to the nearest land — all point-in-polygon work) does not depend on
 * the year and is evaluated once; years year_first .. year_first + n_years - 1 (0 = 2025) differ in the settlements' populations.
 * scores[(site - first_site) * n_years * 15 + y * 15 + type]. The site range [first_site, first_site + n_sites) is what a rank of a
 * sharded run takes; shards need no exchange. HOST output / DEVICE output (asynchronous on the ctx stream). */
int eg_location_analysis_sites(eg_ctx* ctx, int use_loaded_map, uint32_t sites_per_axis, double step, uint32_t year_first,
                               uint32_t n_years, uint32_t first_site, uint32_t n_sites, double* scores_out);
int eg_location_analysis_sites_device(eg_ctx* ctx, int use_loaded_map, uint32_t sites_per_axis, double step, uint32_t year_first,
                                      uint32_t n_years, uint32_t first_site, uint32_t n_sites, double* d_scores);
/* Map::analyze_locations(min_suitability) followed by LocationAnalysis::save_cache(cache_dir) — <cache_dir>/location_analysis.json,
 * the file load_location_analysis reads (map_handler.rs:243-248, core/multi_simulation.rs:149-154) — and save_to_file(text_path), the
 * report of bin/analyze_locations.rs:19-46 (map_handler.rs:208-241). Either path may be NULL. The JSON is
 * serde_json::to_string_pretty of LocationAnalysis (map_handler.rs:48-60): locations, type_counts, multi_type_locations,
 * remaining_spaces, exhausted_types, type_to_locations; the HashMap-typed fields, unordered in the reference, are written in
 * generator-type order. use_loaded_map = 0 is the empty map the reference's tool analyses (the shipped cache). */
int eg_location_analysis_write(eg_ctx* ctx, int use_loaded_map, double min_suitability, const char* cache_dir, const char* text_path);

/* ---- measurement aid (not on the path): double-precision multiply+add issue rate of `device` in TFLOP/s WITHOUT fused
 * multiply-add — the arithmetic ceiling of kernels compiled with --fmad=false like the episode kernel (BASELINE.md §3). */
int eg_microbench_fp64(int device, double* tflops_out);
/* ---- test aid (not on the path): the update rule's shared arithmetic (csrc/eg_math.hpp, csrc/update_rule.hpp), evaluated on
 * the host (device < 0) or on GPU `device`, so that tests can hold the host and the device form to the same bits and to
 * high-precision references. fn: 0 exp(x), 1 ln(x), 2 pow(x, y), 3 score_metrics(net x, opinion 0.5, cost y), 4/5/6 penalty /
 * boost / mild penalty of apply_contrast_learning for (best score 2.0, current score x, stagnation counter y, lr 0.2), 7/8
 * penalty / boost of apply_deficit_contrast_learning for counter y, 9 one draw of the update's Philox stream. */
int eg_rule_math(int device, uint32_t fn, const double* x, const double* y, uint32_t n, double* out);

#ifdef __cplusplus
}
#endif
#endif /* EIRGRID_B200_H */
