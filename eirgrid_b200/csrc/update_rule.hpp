// update_rule.hpp — the scalar part of the reference's per-episode weight update, ONE source for the host form
// (weights.cpp, eg_update) and the device form (update.cu, eg_update_device).
//
// apply_contrast_learning (ai/learning/weights/learning.rs:131-283) and apply_deficit_contrast_learning
// (learning.rs:285-373) turn (best score, this episode's score, iterations_without_improvement, learning rate) into a
// handful of factors — boost, penalty, mild penalty — that are then multiplied into the table entries of the actions
// the episode and the best strategy recorded. Everything up to those factors is here, written once, so that the two
// forms execute the same IEEE operations in the same order (host: -ffp-contract=off, device: --fmad=false) and end with
// the same bits. exp / ln / pow come from eg_math.hpp for the same reason. The weight clamps, the scoring constants and the
// deficit-key order are defined here only: the episode kernel, the batch statistics and the file writers use them too.
#pragma once
#include "eg_math.hpp"
#include "tables.h"

namespace egrule {

constexpr double kMinWeight = 0.0001, kMaxWeight = 0.999;              // ai/learning/constants.rs:14-15
constexpr double kMaxCost = 50000000000.0, kMaxEmissions = 1000000.0;  // config/constants.rs:112-113
constexpr int kContrastDraws = 26 * 61;                                // draws the randomisation branch of learning.rs:267-280 consumes

// std::min / std::max / f64::max as the host form uses them (NaN behaviour included)
EGM_HD double min_std(double a, double b) { return (b < a) ? b : a; }   // std::min(a, b)
EGM_HD double max_std(double a, double b) { return (a < b) ? b : a; }   // std::max(a, b)
EGM_HD double max_nan(double a, double b) {                             // std::fmax / f64::max: the non-NaN operand (quirk Q9)
  if (a != a) return b;
  if (b != b) return a;
  return (a < b) ? b : a;
}

// score_metrics, ai/metrics/scoring.rs:5-45 (m = net emissions, public opinion, total cost, reliability)
EGM_HD double score(const double m[4], bool cost_only) {
  const double normalized_cost = max_std(m[2] / kMaxCost, 1.0);
  const double log_cost = egm::log(normalized_cost);
  const double max_expected_log_cost = egm::log(kMaxCost * 100.0 / kMaxCost);
  if (cost_only) return 2.0 - min_std(log_cost / max_expected_log_cost, 1.0);
  if (m[0] > 0.0) return 1.0 - min_std(m[0] / kMaxEmissions, 1.0);
  const double cost_score = 1.0 - min_std(log_cost / max_expected_log_cost, 1.0);
  const double cost_weight = normalized_cost > 8.0 ? 0.8 : 0.5;
  const double opinion_weight = 1.0 - cost_weight;
  return 1.0 + (cost_score * cost_weight + m[1] * opinion_weight);
}

struct Contrast {   // apply_contrast_learning, learning.rs:131-194 and 267
  bool applied;     // deterioration passed the dynamic threshold, or iterations_without_improvement > 800
  bool randomise;   // iterations_without_improvement > 1200: every weight is multiplied by U(0.75, 1.25) afterwards
  double boost;     // every occurrence of an action in the best strategy
  double penalty;   // every recorded action that the best strategy does not contain
  double mild;      // a recorded action the best strategy holds at another position
};

EGM_HD Contrast contrast(double best_score, double current_score, uint32_t iwi, double learning_rate) {
  Contrast c;
  const double deterioration = best_score > 0.0 ? (best_score - current_score) / best_score : 0.0;
  const double iterations = (double)iwi;
  const double threshold = 0.1 * max_std(egm::exp(-iterations / 500.0), 0.00001 / 0.1);
  const bool force = iwi > 800;
  c.applied = deterioration > threshold || force;
  c.randomise = false;
  c.boost = c.penalty = c.mild = 1.0;
  if (!c.applied) return c;
  const double stagnation = 1.0 + (0.2 * egm::pow((double)iwi / 10.0, 1.8));
  const double combined = egm::pow(deterioration, 0.3) * stagnation;
  const double alr = learning_rate * (1.0 + 0.1 * (double)iwi);
  c.penalty = 1.0 / (1.0 + alr * 1.5 * combined);
  c.boost = 1.0 + (alr * 2.0 * stagnation);
  c.mild = 1.0 / (1.0 + alr * combined * 0.5);
  c.randomise = iwi > 1200;
  return c;
}

// apply_deficit_contrast_learning, learning.rs:285-310 and 358 — called AFTER update_best_strategy, so `iwi` is the
// counter that call left behind (0 for an improving episode: never applied then)
EGM_HD Contrast deficit_contrast(uint32_t iwi, double learning_rate) {
  Contrast c;
  const double deterioration = (double)iwi / 10.0;
  const double threshold = 0.05 * max_std(egm::exp(-(double)iwi / 400.0), 0.00001 / 0.05);
  const bool force = iwi > 800;
  c.applied = deterioration > threshold || force;
  c.randomise = false;
  c.boost = c.penalty = c.mild = 1.0;
  if (!c.applied) return c;
  const double stagnation = 1.0 + (0.2 * egm::pow((double)iwi / 10.0, 1.8));
  const double combined = egm::pow(deterioration, 0.3) * stagnation;
  const double alr = learning_rate * (1.0 + 0.1 * (double)iwi);
  c.penalty = 1.0 / (1.0 + alr * 1.5 * combined);
  c.boost = 1.0 + (alr * 2.0 * stagnation * 1.5);
  c.randomise = iwi > 1200;
  return c;
}

// The randomisation branch draws from a counter-based stream of our own (the reference uses thread_rng there, which no
// run can reproduce): draw d of the episode with iteration counter c is Philox4x32-10(counter = (c, 0, d, "UPDT"),
// key = rng_seed) as a 53-bit uniform.
EGM_HD double update_uniform(uint32_t key_lo, uint32_t key_hi, uint32_t iteration, uint32_t draw) {
  uint32_t x[4] = {iteration, 0u, draw, 0x55504454u};
  egm::philox4x32_10(x, key_lo, key_hi);
  return egm::uniform53(x[0], x[1]);
}

// one randomisation step of a weight: w * (1 + 0.25 * (2u - 1)) clamped like learning.rs:275-277
EGM_HD double random_factor(double u) { return 1.0 + 0.25 * (u * 2.0 - 1.0); }
EGM_HD double apply_random_factor(double w, double f) { return min_std(max_std(w * f, kMinWeight), kMaxWeight); }
EGM_HD double randomise(double w, double u) { return apply_random_factor(w, random_factor(u)); }

// Deficit keys in the insertion order of weights/core.rs:130-152: key k < 14 is AddGenerator(kDeficitKeyTypes[k], 100 %),
// key 14 is DoNothing.
constexpr int kDeficitKeyTypes[14] = {8, 7, 12, 11, 9, 0, 1, 4, 10, 5, 2, 3, 13, 14};

// The same order as 4-bit fields of one word each, for branch-free lookups: the type of key k, and the key of type t
// (0xF: CoalPlant, the one type without a key).
constexpr uint64_t pack_types_of_keys() {
  uint64_t v = 0;
  for (int k = 0; k < 14; k++) v |= (uint64_t)kDeficitKeyTypes[k] << (4 * k);
  return v;
}
constexpr uint64_t pack_keys_of_types() {
  uint64_t v = (1ull << (4 * EG_NT)) - 1;
  for (int k = 0; k < 14; k++) v ^= (uint64_t)(0xF ^ k) << (4 * kDeficitKeyTypes[k]);
  return v;
}
constexpr uint64_t kTypeOfKey = pack_types_of_keys(), kKeyOfType = pack_keys_of_types();

// action code of deficit key k (k >= 14: DoNothing)
EGM_HD int deficit_key_action(uint32_t k) { return k < 14 ? 3 * (int)((kTypeOfKey >> (4 * k)) & 0xF) : EG_ACT_DO_NOTHING; }

// deficit key of an action code, -1 if the action is not a deficit key
EGM_HD int deficit_key_of_action(int code) {
  if (code == EG_ACT_DO_NOTHING) return 14;
  if ((unsigned)code >= 45u || code % 3) return -1;
  const int k = (int)((kKeyOfType >> (4 * (code / 3))) & 0xF);
  return k == 0xF ? -1 : k;
}

}  // namespace egrule
