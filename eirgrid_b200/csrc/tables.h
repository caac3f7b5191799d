// tables.h — layout of the static tables the episode kernels read (HBM-resident, built once per map).
//
// Everything that needs libm (pow/exp) is tabulated on the host from small integer arguments
// (year offsets), so the device path needs only + - * / sqrt, which are IEEE-exact in CUDA when the
// kernels are compiled with --fmad=false. That is what makes results bit-comparable with the
// CPU restatement of the reference (DESIGN.md §numerics).
#pragma once
#include <stdint.h>
#include "../../include/eirgrid_b200.h"

#define EG_NY EG_N_YEARS
#define EG_NT EG_N_GEN_TYPES
#define EG_N_RCLASS 6   // placement penalty radii 3,5,6,7,8,12 km (gpu/metal_location_search.rs:139-146)
#define EG_N_PCLASS 7   // (radius, needs-coast-factor) combinations that occur among the 15 types
// largest distance/radius factor table (all radius classes, each ending with its 1.0) of the forms that copy it into shared memory
// (EgDeviceMap::near_geom); the episode kernel's block shapes are sized for them
#define EG_COMPACT_MAX_FACTORS 2048  // compact form
#define EG_MEDIUM_MAX_FACTORS 5600   // medium form

// generation accumulator a plant's output is added to (map_handler.rs:852-865)
enum { EG_ACC_PLAIN = 0, EG_ACC_INTERMITTENT = 1, EG_ACC_STORAGE = 2 };

struct EgYearRow {       // one per simulated year
  double usage_total;    // calc_total_power_usage(year)                      map_handler.rs:819-827
  double inflation;      // calc_inflation_factor(year)                       const_funcs.rs:13-15
  double carbon_price;   // carbon_price(year)                                const_funcs.rs:186-203
  // sequential accumulators after the existing plants (they come first in Map.generators)
  double ex_gen[3];      // plain / intermittent / storage generation         map_handler.rs:852-865
  double ex_co2;         // calc_total_co2_emissions prefix                   map_handler.rs:902-910
  double ex_opinion_sum; // calculate_average_opinion prefix                  metrics_calculation.rs:7-30
  uint32_t ex_active;    // active existing plants
  uint32_t pop_total;    // calc_total_population                             map_handler.rs:813-817
  uint32_t prefix_changed;  // ex_gen / ex_co2 differ from the previous year's (existing plants came online)
  uint32_t pad;
};

struct EgSmallTables {   // ~35 KB, read-mostly, L1/L2 resident
  EgYearRow year[EG_NY];
  double net_mw[EG_NT];            // get_current_power_output of a new plant           generator.rs:523-554
  double co2[EG_NT];               // get_co2_output of a new plant                     generator.rs:618-626
  double loc_mod[EG_NT];           // location modifier used by get_current_cost        generator.rs:582-594
  double mult[EG_N_MULTS];         // construction_cost_multiplier                      actions.rs:44-45
  double base_cost[EG_NT][EG_NY];  // get_base_cost(build year)                         generator.rs:244-298
  double tech[EG_NT][EG_NY];       // cost_evolution_rate^(year-2025)                   const_funcs.rs:33-34
  double op_type[EG_NY][EG_NT];    // PUBLIC_OPINION_WEIGHT * calc_type_opinion         map_handler.rs:943-947
  double off_amount[EG_N_OFFSET_TYPES];   // base_offset * capture_efficiency           carbon_offset.rs:212-232
  double off_base_cost[EG_N_OFFSET_TYPES];
  double maturity[EG_NY];          // clamp(1-exp(-0.1*d)) for d years since completion carbon_offset.rs:224-228
  double size_factor;              // 1.0 - (size_penalty as f64 * 0.1)                 metal_location_search.rs:166
  uint8_t acc_class[EG_NT];
  uint8_t pclass[EG_NT];           // placement class of the type
  uint8_t rclass_of_pclass[EG_N_PCLASS];
  uint8_t water_of_pclass[EG_N_PCLASS];
  uint8_t natural_offset[EG_N_OFFSET_TYPES];  // Forest/Wetland mature over time
  uint8_t pad[3];
  // what a new plant of the type adds to the (plain, intermittent, storage) generation sums and to the CO2 sum: net_mw in the
  // slot of acc_class, +0.0 in the other two, co2 (read as two 16-byte words)
  alignas(16) double type_sums[EG_NT][4];
  // what the placement walk needs per type, one 8-byte read: [0] = pclass | rclass << 4 | water << 8 | (first entry of the radius
  // class in the block-shared factor table, r2_limit[6 + rclass]) << 16, [1] = r2_limit[rclass]
  alignas(8) uint32_t place_info[EG_NT][2];
};

// per simulation-built plant and year, two doubles:
//   [0] CONSTRUCTION_COST_WEIGHT * calc_cost_opinion(get_current_cost(year), year)   map_handler.rs:944-948
//   [1] get_current_cost(year) = base_cost * inflation * technology factor * location modifier * multiplier
//                                                                                     const_funcs.rs:28-57, generator.rs:582-594
// index [year][type][mult][build year]
#define EG_OPC_INDEX(y, t, m, b) ((((y) * EG_NT + (t)) * EG_N_MULTS + (m)) * EG_NY + (b))
#define EG_OPC_SIZE (EG_NY * EG_NT * EG_N_MULTS * EG_NY)

struct EgDeviceMap {      // device pointers + sizes, passed by value to the kernels
  const EgSmallTables* small;
  const double* plant_terms;      // [EG_OPC_SIZE][2] (cost opinion term, current cost)
  const double* site_opinion;     // [n_sites] avg_settlement_opinion of a plant on the site  map_handler.rs:931-941
  const double* coast_factor;     // [n_sites] 1/(1+min_coast_distance/5000)                  metal_location_search.rs:157-162
  // placement lists, sorted by static score (descending, ties by scan order), per (pclass, year)
  const uint16_t* order;          // [7][26][n_sites] candidate site as (i << 8) | j
  const void* unused[2];          // read by no kernel, but without these 16 bytes `order` and `walk` share one 16-byte constant
                                  // load and the episode kernels compile to a different instruction schedule
  const double* walk;             // [7][26][n_sites][2] (static score, prefix score) of the sorted site, what the placement walk reads
  const double* near_factor;      // [6][r2_stride] distance/radius by squared cell distance d2 (valid for d2 < r2_limit[rc])
  const int* r2_limit;            // [6] first squared cell distance that is NOT inside the penalty radius, followed by
                                  // [6] start of the class in the compact table (prefix sums of the limits) and [1] its size
  int r2_stride;
  int n_sites;
  int grid_n;
  int kmax;                       // plants farther than kmax-1 cells (in x or y) are outside every radius
  int near_geom;                  // which form of the cell-distance arithmetic the episode kernel uses: 0 compact (at most 64 sites
                                  // per axis: one IDP.4A per site and plant), 1 medium (at most 181: IDP.2A + add; both read the
                                  // factors from a block-shared copy of the table), 2 general (coordinates up to 255 or a factor
                                  // table too large for shared memory: plain integer cell distances, table in global memory)
};

#define EG_POLICY_ROW (EG_N_ACTIONS + EG_N_DEFICIT_KEYS + EG_N_COUNT_KEYS + 1)  // 98 doubles = 784 bytes, a multiple of 16

struct EgPolicyDevice {   // weights snapshot + the per-batch constants of update_weights (learning.rs:36-55)
  // one contiguous row per year: [61 regular | 15 deficit | 21 count weights | pad] — what an episode copies into its
  // private buffer with 16-byte asynchronous copies at the start of the year
  double rows[EG_NY][EG_POLICY_ROW];
  double learning_rate;
  double exploration_rate;
  double action_exploration;      // sample_action's rate: exploration_rate / (1 + 0.01 iwi) once iwi > 100 (sampling.rs:150-156)
  double relative_improvement;    // learning.rs:40-49 (0 whenever a best strategy with positive score exists)
  // stagnation branch of sample_action (sampling.rs:190-220), evaluated per snapshot with the host libm
  double stagnation_power;        // 1 + 2 * min(iwi / 1000, 3)
  double w_total[EG_NY];          // left-to-right sums of the rows, as sample_action / sample_deficit_action /
  double dw_total[EG_NY];         // sample_additional_actions compute them (sampling.rs:182,352-355,406)
  double cw_total[EG_NY];
  double scaled_sorted[EG_NY][EG_N_ACTIONS];  // weight^power in stable descending weight order
  double scaled_total[EG_NY];     // their left-to-right sums (sampling.rs:199)
  uint32_t iwi;                   // iterations_without_improvement
  uint32_t has_count_weights;
  uint32_t noop_boost;            // learning.rs:82: best is net-zero but costs > 8 * MAX_ACCEPTABLE_COST
  uint32_t has_best;
  // best strategy for replay iterations (force_best_actions, sampling.rs:78-145,242-313)
  // (lists of any length on the host; here back to back, year after year, like the rows of eg_traj)
  uint16_t n_best[EG_NY];            // len(best_actions[y])
  uint16_t n_best_deficit[EG_NY];    // len(best_deficit_actions[y])
  uint16_t best_off[EG_NY];          // start of year y's list in best[]
  uint16_t best_deficit_off[EG_NY];  // start of year y's list in best_deficit[]
  uint8_t best[EG_BEST_CAPACITY];
  uint8_t best_deficit[EG_TRAJ_CAPACITY];
  uint8_t sorted_idx[EG_NY][64];  // action code at each rank of scaled_sorted
};
