// weights.hpp — host-side policy table (the reference's ActionWeights, ai/learning/weights/mod.rs:49-107)
// stored densely: 26 years x (61 action keys, 15 deficit keys, 21 count keys).
#pragma once
#include <cstdint>
#include <string>
#include <vector>
#include "tables.h"

struct EgImprovement {  // utils/csv_export.rs ImprovementRecord as serialised by ai/learning/serialization.rs:10-19
  uint32_t iteration;
  double score, net_emissions, total_cost, public_opinion, power_reliability;
  std::string timestamp;
};

struct eg_weights {
  double w[EG_NY][EG_N_ACTIONS];
  double dw[EG_NY][EG_N_DEFICIT_KEYS];
  double cw[EG_NY][EG_N_COUNT_KEYS];
  bool has_count_weights = true;
  double learning_rate = 0.2;      // DEFAULT_LEARNING_RATE
  double exploration_rate = 0.2;   // DEFAULT_EXPLORATION_RATE
  bool has_best = false;
  double best_metrics[4] = {0, 0, 0, 0};  // net emissions, opinion, total cost, reliability
  std::vector<double> best_weights;       // 26*61 when has_best
  std::vector<uint8_t> best_actions[EG_NY];
  std::vector<uint8_t> best_deficit_actions[EG_NY];
  uint32_t iteration_count = 0;
  uint32_t iwi = 0;                // iterations_without_improvement
  std::string optimization_mode;   // "" == None (never set by the reference driver, quirk Q12)
  std::vector<EgImprovement> history;
  eg_weights();
};

// names the reference prints for the parts of an action key: GeneratorType and CarbonOffsetType variants in key order, cost
// multipliers in percent
constexpr const char* kGenNames[EG_NT] = {"OnshoreWind", "OffshoreWind", "DomesticSolar", "CommercialSolar", "UtilitySolar",
                                          "Nuclear", "CoalPlant", "GasCombinedCycle", "GasPeaker", "Biomass", "HydroDam",
                                          "PumpedStorage", "BatteryStorage", "TidalGenerator", "WaveEnergy"};
constexpr const char* kOffsetNames[EG_N_OFFSET_TYPES] = {"Forest", "Wetland", "ActiveCapture", "CarbonCredit"};
constexpr int kMultPercent[EG_N_MULTS] = {100, 120, 150};
// an action code as the reference prints the GridAction (impl Display, ai/actions/grid_action.rs:18-41)
std::string eg_action_display(int code);

// fills the device-side snapshot (weights + per-batch constants of update_weights + best lists); false when the best
// lists are longer than the snapshot's capacity (EG_BEST_CAPACITY / EG_TRAJ_CAPACITY slots) and were cut
bool eg_weights_fill_policy(const eg_weights& w, EgPolicyDevice* out);

// per-batch constants of the batch-synchronous contrast rule, shared by the stats kernel and the host apply
struct EgContrastConsts {
  uint32_t has_best;
  uint32_t force;            // iwi > 800
  uint32_t cost_only;        // the weights' own optimization_mode is "cost_only" (only ever set by a checkpoint file, quirk Q12)
  uint32_t pad;
  double best_score;
  double threshold;          // 0.1 * max(exp(-iwi/500), 1e-4)
  double stagnation;         // 1 + 0.2 * (iwi/10)^1.8
  double alr;                // lr * (1 + 0.1 * iwi)
  double boost;              // 1 + alr * 2 * stagnation
};
EgContrastConsts eg_contrast_consts(const eg_weights& w);

// host <-> device marshalling of the in-order device update (update.cu): fill = the fields of `w` the rule touches plus its
// best strategy as slot 0 (false: the lists exceed EG_UPD_CAT_CAPACITY); apply = the state after the passes back into `w`,
// with one improvement_history entry per improving episode (iteration0 = w.iteration_count before the call)
struct EgUpdState;
struct EgUpdSlot;
struct EgUpdImprovement;
bool eg_weights_fill_update_state(const eg_weights& w, EgUpdState* st, EgUpdSlot* slot0);
void eg_weights_apply_update_state(eg_weights& w, const EgUpdState& st, const EgUpdSlot& slot0, const EgUpdImprovement* improvements,
                                   uint32_t n_improvements, uint32_t iteration0);

#define EG_STATS_FIXED_SCALE 16777216.0  // 2^24: fixed-point scale of the summed log-factors
#define EG_STATS_YEAR_STRIDE (3 * EG_N_ACTIONS + EG_N_DEFICIT_KEYS)
#define EG_STATS_HEADER 8
