// weights.cpp — host side of the policy table: construction, JSON checkpoints, merge and the weight update.
//
// Replaces ActionWeights::new (ai/learning/weights/core.rs:25-250), save_to_file / load_from_file
// (weights/serialization.rs:29-493, schema ai/learning/serialization.rs:37-51), update_weights_from
// (weights/strategy.rs:281-311) and the write-lock section of the batch driver, core/multi_simulation.rs:494-508:
// transfer_recorded_actions_from -> apply_contrast_learning -> update_best_strategy -> apply_deficit_contrast_learning
// (weights/strategy.rs:313-342,19-258; weights/learning.rs:131-373).
// HashMap<GridAction, f64> becomes a dense row in canonical key order (see include/eirgrid_b200.h).
#include "weights.hpp"
#include "json_min.hpp"
#include "common.hpp"
#include "update_rule.hpp"
#include "update.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <ctime>

namespace {

using egrule::deficit_key_action;
using egrule::deficit_key_of_action;
using egrule::kMaxWeight;
using egrule::kMinWeight;

// score_metrics(metrics, self.optimization_mode) as the weights object itself scores (learning.rs:134-135, strategy.rs:20,58):
// the mode only ever comes from a checkpoint file, the reference's driver never sets it (quirk Q12)
double score_w(const eg_weights& W, const double m[4]) { return egrule::score(m, W.optimization_mode == "cost_only"); }

bool contains(const std::vector<uint8_t>& v, uint8_t a) { return std::find(v.begin(), v.end(), a) != v.end(); }

// ---- JSON <-> action code ---------------------------------------------------------------------------------
std::string render_action(int code, const std::string& ind) {
  // SerializableAction, ai/actions/serializable_action.rs:6-13 (field order of the struct)
  const char* type = "DoNothing";
  std::string gen = "null", id = "null", pct = "null", off = "null", mult = "null";
  if (code < 45) { type = "AddGenerator"; gen = std::string("\"") + kGenNames[code / 3] + "\""; mult = std::to_string(kMultPercent[code % 3]); }
  else if (code < 57) { type = "AddCarbonOffset"; off = std::string("\"") + kOffsetNames[(code - 45) / 3] + "\""; mult = std::to_string(kMultPercent[(code - 45) % 3]); }
  else if (code == EG_ACT_UPGRADE) { type = "UpgradeEfficiency"; id = "\"\""; }
  else if (code == EG_ACT_ADJUST) { type = "AdjustOperation"; id = "\"\""; pct = "0"; }
  else if (code == EG_ACT_CLOSE) { type = "CloseGenerator"; id = "\"\""; }
  std::string o;
  o += ind + "{\n";
  o += ind + "  \"action_type\": \"" + type + "\",\n";
  o += ind + "  \"generator_type\": " + gen + ",\n";
  o += ind + "  \"generator_id\": " + id + ",\n";
  o += ind + "  \"operation_percentage\": " + pct + ",\n";
  o += ind + "  \"offset_type\": " + off + ",\n";
  o += ind + "  \"cost_multiplier\": " + mult + "\n";
  o += ind + "}";
  return o;
}

// a checkpoint holds ~3,600 action objects out of 61 different ones at two indentations: each text is rendered once
void write_action(std::string& o, int code, const std::string& ind) {
  static std::string cache[2][EG_N_ACTIONS];
  static bool ready = false;
  static const std::string kInd[2] = {"        ", "      "};
  if (!ready) {
    for (int i = 0; i < 2; i++)
      for (int c = 0; c < EG_N_ACTIONS; c++) cache[i][c] = render_action(c, kInd[i]);
    ready = true;
  }
  for (int i = 0; i < 2; i++)
    if (ind == kInd[i] && code >= 0 && code < EG_N_ACTIONS) { o += cache[i][code]; return; }
  o += render_action(code, ind);
}

// a JSON number as the u32 the reference's struct declares (serde fails the load on anything else); a missing or null
// value keeps the default
bool number_as_u32(const egjson::Value* v, uint32_t* out) {
  if (!v || v->is_null()) return true;
  if (v->kind != egjson::Value::Number || !(v->num >= 0.0 && v->num <= 4294967295.0) || v->num != std::floor(v->num)) return false;
  *out = (uint32_t)v->num;
  return true;
}

// returns the action code or -1 for keys outside the closed key set (e.g. a 200 % multiplier)
int read_action(const egjson::Value& v) {
  const egjson::Value* type = v.get("action_type");
  if (!type || type->kind != egjson::Value::String) return -1;
  auto mult_index = [&]() {
    const egjson::Value* m = v.get("cost_multiplier");
    int pct = (m && m->kind == egjson::Value::Number && m->num >= 0.0 && m->num <= 65535.0) ? (int)m->num : 100;  // unwrap_or(DEFAULT_COST_MULTIPLIER); u16
    for (int i = 0; i < EG_N_MULTS; i++)
      if (kMultPercent[i] == pct) return i;
    return -1;
  };
  if (type->str == "AddGenerator") {
    const egjson::Value* g = v.get("generator_type");
    int t = 8;  // GasPeaker when the type is missing (weights/serialization.rs:163)
    if (g && g->kind == egjson::Value::String) {
      t = -1;
      for (int i = 0; i < EG_NT; i++)
        if (g->str == kGenNames[i]) t = i;
      if (t < 0) return -3;  // unknown generator type: an error in the main table, skipped elsewhere
    }
    int m = mult_index();
    return m < 0 ? -1 : 3 * t + m;
  }
  if (type->str == "AddCarbonOffset") {
    const egjson::Value* o = v.get("offset_type");
    int ot = 0;  // Forest for unknown names (weights/serialization.rs:185)
    if (o && o->kind == egjson::Value::String)
      for (int i = 0; i < EG_N_OFFSET_TYPES; i++)
        if (o->str == kOffsetNames[i]) ot = i;
    int m = mult_index();
    return m < 0 ? -1 : 45 + 3 * ot + m;
  }
  if (type->str == "UpgradeEfficiency") return EG_ACT_UPGRADE;
  if (type->str == "AdjustOperation") return EG_ACT_ADJUST;
  if (type->str == "CloseGenerator") return EG_ACT_CLOSE;
  if (type->str == "DoNothing") return EG_ACT_DO_NOTHING;
  return -2;  // unknown action type: load_from_file fails with InvalidData
}

void write_weight_map(std::string& o, const char* name, const double* rows, int n_keys, bool deficit, bool present) {
  o += std::string("  \"") + name + "\": ";
  if (!present) { o += "null"; return; }
  o += "{\n";
  for (int y = 0; y < EG_NY; y++) {
    o += "    \"" + std::to_string(EG_BASE_YEAR + y) + "\": [\n";
    for (int k = 0; k < n_keys; k++) {
      int code = deficit ? deficit_key_action(k) : k;
      o += "      [\n";
      write_action(o, code, "        ");
      o += ",\n        " + egjson::fmt_double(rows[(size_t)y * n_keys + k]) + "\n      ]";
      o += k + 1 < n_keys ? ",\n" : "\n";
    }
    o += y + 1 < EG_NY ? "    ],\n" : "    ]\n";
  }
  o += "  }";
}

void write_action_lists(std::string& o, const char* name, const std::vector<uint8_t>* lists, bool present) {
  o += std::string("  \"") + name + "\": ";
  if (!present) { o += "null"; return; }
  o += "{\n";
  for (int y = 0; y < EG_NY; y++) {
    o += "    \"" + std::to_string(EG_BASE_YEAR + y) + "\": [";
    if (!lists[y].empty()) {
      o += "\n";
      for (size_t i = 0; i < lists[y].size(); i++) {
        write_action(o, lists[y][i], "      ");
        o += i + 1 < lists[y].size() ? ",\n" : "\n";
      }
      o += "    ]";
    } else {
      o += "]";
    }
    o += y + 1 < EG_NY ? ",\n" : "\n";
  }
  o += "  }";
}

// year keys are u32 in the reference's maps (HashMap<u32, _>): anything else fails the whole load there
bool parse_year_key(const std::string& k, long long* year) {
  if (k.empty() || k.size() > 10) return false;
  for (char ch : k)
    if (ch < '0' || ch > '9') return false;
  *year = std::atoll(k.c_str());
  return *year <= 4294967295ll;
}

bool read_weight_map(const egjson::Value* v, double* rows, int n_keys, bool deficit, bool* any) {
  if (!v || v->kind != egjson::Value::Object) return true;
  for (const auto& kv : v->obj) {
    long long year = 0;
    if (!parse_year_key(kv.first, &year)) return false;
    if (year < EG_BASE_YEAR || year > EG_END_YEAR || kv.second.kind != egjson::Value::Array) continue;
    for (const egjson::Value& entry : kv.second.arr) {
      if (entry.kind != egjson::Value::Array || entry.arr.size() != 2) continue;
      int code = read_action(entry.arr[0]);
      if ((code == -2 || code == -3) && !deficit) return false;  // weights/serialization.rs:158-159,201-205
      if (code < 0) continue;
      int k = deficit ? deficit_key_of_action(code) : code;
      if (k < 0 || k >= n_keys) continue;
      rows[(size_t)(year - EG_BASE_YEAR) * n_keys + k] = entry.arr[1].num;
      if (any) *any = true;
    }
  }
  return true;
}

bool read_action_lists(const egjson::Value* v, std::vector<uint8_t>* lists) {
  if (!v || v->kind != egjson::Value::Object) return true;
  for (const auto& kv : v->obj) {
    long long year = 0;
    if (!parse_year_key(kv.first, &year)) return false;
    if (year < EG_BASE_YEAR || year > EG_END_YEAR || kv.second.kind != egjson::Value::Array) continue;
    for (const egjson::Value& a : kv.second.arr) {
      int code = read_action(a);
      if (code >= 0) lists[year - EG_BASE_YEAR].push_back((uint8_t)code);
    }
  }
  return true;
}

// the episode's recorded lists as the shared weights see them after transfer_recorded_actions_from
struct Recorded {
  std::vector<uint8_t> run[EG_NY], deficit[EG_NY];
  void from_traj(const eg_traj& t, bool replay) {
    int row = 0;  // the year rows follow each other in the record; counts that run past its capacity are cut
    for (int y = 0; y < EG_NY; y++) {
      run[y].clear();
      deficit[y].clear();
      const int nd = std::min<int>(t.n_deficit[y], EG_TRAJ_CAPACITY - row);
      const int na = std::min<int>(t.n_additional[y], EG_TRAJ_CAPACITY - row - nd);
      const uint8_t* a = t.actions + row;
      // replay iterations record every sampled action twice (sampling.rs:97-99,262-264 + simulation.rs:197,406-409; quirk Q10)
      // (codes outside the key set never come from the device; a malformed record must not index the tables with them)
      for (int i = 0; i < nd; i++) {
        if (a[i] >= EG_N_ACTIONS) continue;
        run[y].push_back(a[i]);
        deficit[y].push_back(a[i]);
        if (replay && i < 4) deficit[y].push_back(a[i]);
      }
      for (int i = nd; i < nd + na; i++) {
        if (a[i] >= EG_N_ACTIONS) continue;
        run[y].push_back(a[i]);
        if (replay) run[y].push_back(a[i]);
      }
      row += nd + na;
    }
  }
};

struct UpdateRng {  // the stream of the randomisation branch (learning.rs:267-280,358-370): egrule::update_uniform's draws in order
  uint32_t k0, k1, iteration, draw;
  double f64() { return egrule::update_uniform(k0, k1, iteration, draw++); }
};

void contrast(eg_weights& W, const Recorded& rec, const double metrics[4], UpdateRng* rng, uint32_t* applied) {  // learning.rs:131-283
  if (!W.has_best) return;
  // thresholds and factors: update_rule.hpp, the source the device form (update.cu) shares
  const egrule::Contrast c = egrule::contrast(score_w(W, W.best_metrics), score_w(W, metrics), W.iwi, W.learning_rate);
  if (!c.applied) return;
  if (applied) (*applied)++;
  for (int y = 0; y < EG_NY; y++) {
    std::vector<uint8_t> cur = rec.run[y];
    cur.insert(cur.end(), rec.deficit[y].begin(), rec.deficit[y].end());
    std::vector<uint8_t> best = W.best_actions[y];
    best.insert(best.end(), W.best_deficit_actions[y].begin(), W.best_deficit_actions[y].end());
    double* row = W.w[y];
    for (uint8_t a : best) row[a] = std::min(row[a] * c.boost, kMaxWeight);
    for (size_t i = 0; i < cur.size(); i++) {
      const uint8_t a = cur[i];
      if (!contains(best, a)) {
        row[a] = std::fmax(row[a] * c.penalty, kMinWeight);  // NaN penalty collapses to MIN_WEIGHT like f64::max (quirk Q9)
      } else if (i < best.size() && a != best[i]) {
        row[a] = std::fmax(row[a] * c.mild, kMinWeight);
      }
    }
  }
  if (c.randomise && rng)
    for (int y = 0; y < EG_NY; y++)
      for (int k = 0; k < EG_N_ACTIONS; k++) W.w[y][k] = egrule::randomise(W.w[y][k], rng->f64());
}

std::string now_string() {
  char buf[32];
  std::time_t t = std::time(nullptr);
  std::tm tmv;
  localtime_r(&t, &tmv);
  std::strftime(buf, sizeof(buf), "%Y-%m-%d %H:%M:%S", &tmv);
  return buf;
}

// The episodes `imps` (numbered from iteration0) improved on the best strategy one after the other (strategy.rs:26-50): each
// gets its improvement_history entry, all with one timestamp, and the last one becomes the best strategy, with the weight
// table `weights` and the action lists `lists` it was recorded with.
void record_best(eg_weights& W, const EgUpdImprovement* imps, uint32_t n, uint32_t iteration0, const double* weights, const Recorded& lists) {
  const std::string now = now_string();
  for (uint32_t i = 0; i < n; i++) {
    const EgUpdImprovement& r = imps[i];
    W.history.push_back({iteration0 + (uint32_t)r.episode + 1u, r.score, r.metrics[0], r.metrics[2], r.metrics[1], r.metrics[3], now});
  }
  std::memcpy(W.best_metrics, imps[n - 1].metrics, sizeof(W.best_metrics));
  W.has_best = true;
  W.best_weights.assign(weights, weights + EG_NY * EG_N_ACTIONS);
  for (int y = 0; y < EG_NY; y++) {
    W.best_actions[y] = lists.run[y];
    W.best_deficit_actions[y] = lists.deficit[y];
  }
}

bool best_strategy(eg_weights& W, const Recorded& rec, const double metrics[4]) {  // strategy.rs:19-258
  const double current_score = score_w(W, metrics);
  const bool should_update = !W.has_best || current_score > score_w(W, W.best_metrics);
  if (should_update) {
    const EgUpdImprovement imp{0, current_score, {metrics[0], metrics[1], metrics[2], metrics[3]}};
    record_best(W, &imp, 1, W.iteration_count, &W.w[0][0], rec);
  }
  W.iteration_count += 1;
  W.iwi = should_update ? 0 : W.iwi + 1;
  return should_update;
}

void deficit_contrast(eg_weights& W, const Recorded& rec, UpdateRng* rng) {  // learning.rs:285-373
  if (!W.has_best) return;
  const egrule::Contrast c = egrule::deficit_contrast(W.iwi, W.learning_rate);
  if (!c.applied) return;
  for (int y = 0; y < EG_NY; y++) {
    const std::vector<uint8_t>& best = W.best_deficit_actions[y];
    double* row = W.dw[y];
    for (uint8_t a : best) {
      int k = deficit_key_of_action(a);
      if (k >= 0) row[k] = std::min(row[k] * c.boost, kMaxWeight);
    }
    for (uint8_t a : rec.deficit[y])
      if (!contains(best, a)) {
        int k = deficit_key_of_action(a);
        if (k >= 0) row[k] = std::fmax(row[k] * c.penalty, kMinWeight);
      }
  }
  if (c.randomise && rng)
    for (int y = 0; y < EG_NY; y++)
      for (int k = 0; k < EG_N_DEFICIT_KEYS; k++) W.dw[y][k] = egrule::randomise(W.dw[y][k], rng->f64());
}

}  // namespace

eg_weights::eg_weights() {  // ActionWeights::new, weights/core.rs:25-250
  static const double gw[EG_NT] = {0.08, 0.08, 0.05, 0.05, 0.08, 0.03, 0.04, 0.06, 0.02, 0.04, 0.06, 0.06, 0.07, 0.05, 0.05};
  static const double dk[EG_N_DEFICIT_KEYS] = {0.15, 0.15, 0.15, 0.10, 0.10, 0.07, 0.07, 0.06, 0.06, 0.05, 0.01, 0.01, 0.01, 0.01, 0.001};
  for (int y = 0; y < EG_NY; y++) {
    for (int t = 0; t < EG_NT; t++) {
      w[y][3 * t] = gw[t];
      w[y][3 * t + 1] = gw[t] * 0.5;
      w[y][3 * t + 2] = gw[t] * 0.25;
    }
    for (int o = 0; o < EG_N_OFFSET_TYPES; o++) {
      w[y][45 + 3 * o] = 0.02;
      w[y][45 + 3 * o + 1] = 0.02 * 0.5;
      w[y][45 + 3 * o + 2] = 0.02 * 0.25;
    }
    w[y][EG_ACT_UPGRADE] = 0.04;
    w[y][EG_ACT_ADJUST] = 0.04;
    w[y][EG_ACT_CLOSE] = 0.02;
    w[y][EG_ACT_DO_NOTHING] = 0.1;
    for (int k = 0; k < EG_N_DEFICIT_KEYS; k++) dw[y][k] = dk[k];
    double total = 0.0;
    for (int c = 0; c < EG_N_COUNT_KEYS; c++) {
      const double base = std::exp(-0.8 * (double)c);
      const double bias = c == 0 ? 4.0 : c == 1 ? 3.5 : c == 2 ? 3.0 : c == 3 ? 2.5 : c == 4 ? 2.0 : c == 5 ? 1.5 : 1.0;
      cw[y][c] = base * bias;
      total += cw[y][c];
    }
    for (int c = 0; c < EG_N_COUNT_KEYS; c++) cw[y][c] /= total;
  }
}

bool eg_weights_fill_policy(const eg_weights& W, EgPolicyDevice* out) {
  std::memset(out, 0, sizeof(*out));
  for (int y = 0; y < EG_NY; y++) {
    std::memcpy(&out->rows[y][0], W.w[y], sizeof(W.w[y]));
    std::memcpy(&out->rows[y][EG_N_ACTIONS], W.dw[y], sizeof(W.dw[y]));
    std::memcpy(&out->rows[y][EG_N_ACTIONS + EG_N_DEFICIT_KEYS], W.cw[y], sizeof(W.cw[y]));
  }
  out->learning_rate = W.learning_rate;
  out->exploration_rate = W.exploration_rate;
  out->action_exploration = W.iwi > 100 ? W.exploration_rate * (1.0 / (1.0 + 0.01 * (double)W.iwi)) : W.exploration_rate;
  // update_weights (learning.rs:36-49): final_impact_score and best_score are both score(best_metrics)
  double rel = 0.0;
  if (W.has_best) {
    const double best_score = score_w(W, W.best_metrics);
    rel = best_score > 0.0 ? (best_score - best_score) / best_score : best_score;
  }
  out->relative_improvement = rel;
  out->stagnation_power = 1.0 + (2.0 * std::min((double)W.iwi / 1000.0, 3.0));
  for (int y = 0; y < EG_NY; y++) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int k = 0; k < EG_N_ACTIONS; k++) a += W.w[y][k];
    for (int k = 0; k < 14; k++) b += W.dw[y][k];  // AddGenerator keys only (sampling.rs:352-355)
    for (int k = 0; k < EG_N_COUNT_KEYS; k++) c += W.cw[y][k];
    out->w_total[y] = a; out->dw_total[y] = b; out->cw_total[y] = c;
  }
  if (W.iwi > 500) {
    for (int y = 0; y < EG_NY; y++) {
      int idx[EG_N_ACTIONS];
      for (int k = 0; k < EG_N_ACTIONS; k++) idx[k] = k;
      std::stable_sort(idx, idx + EG_N_ACTIONS, [&](int a, int b) { return W.w[y][a] > W.w[y][b]; });
      for (int k = 0; k < EG_N_ACTIONS; k++) {
        out->sorted_idx[y][k] = (uint8_t)idx[k];
        out->scaled_sorted[y][k] = std::pow(W.w[y][idx[k]], out->stagnation_power);
      }
      double t = 0.0;
      for (int k = 0; k < EG_N_ACTIONS; k++) t += out->scaled_sorted[y][k];
      out->scaled_total[y] = t;
    }
  }
  out->iwi = W.iwi;
  out->has_count_weights = W.has_count_weights ? 1 : 0;
  out->noop_boost = (W.has_best && W.best_metrics[0] <= 0.0 && W.best_metrics[2] > egrule::kMaxCost * 8.0) ? 1 : 0;
  out->has_best = W.has_best ? 1 : 0;
  size_t ob = 0, obd = 0;
  bool fits = true;
  for (int y = 0; y < EG_NY; y++) {
    const size_t nb = std::min<size_t>(W.best_actions[y].size(), EG_BEST_CAPACITY - ob);
    const size_t nbd = std::min<size_t>(W.best_deficit_actions[y].size(), EG_TRAJ_CAPACITY - obd);
    fits = fits && nb == W.best_actions[y].size() && nbd == W.best_deficit_actions[y].size();
    out->n_best[y] = (uint16_t)nb; out->best_off[y] = (uint16_t)ob;
    out->n_best_deficit[y] = (uint16_t)nbd; out->best_deficit_off[y] = (uint16_t)obd;
    for (size_t i = 0; i < nb; i++) out->best[ob + i] = W.best_actions[y][i];
    for (size_t i = 0; i < nbd; i++) out->best_deficit[obd + i] = W.best_deficit_actions[y][i];
    ob += nb; obd += nbd;
  }
  return fits;
}

bool eg_weights_fill_update_state(const eg_weights& W, EgUpdState* st, EgUpdSlot* slot0) {
  std::memset(st, 0, sizeof(*st));
  std::memset(slot0, 0, sizeof(*slot0));
  std::memcpy(st->w, W.w, sizeof(st->w));
  std::memcpy(st->dw, W.dw, sizeof(st->dw));
  if (W.best_weights.size() == (size_t)EG_NY * EG_N_ACTIONS) std::memcpy(st->best_w, W.best_weights.data(), sizeof(st->best_w));
  std::memcpy(st->best_metrics, W.best_metrics, sizeof(st->best_metrics));
  st->best_score = W.has_best ? score_w(W, W.best_metrics) : 0.0;
  st->cost_only = W.optimization_mode == "cost_only" ? 1u : 0u;
  st->learning_rate = W.learning_rate;
  st->batch_best_index = -1;
  st->has_best = W.has_best ? 1u : 0u;
  st->iwi = W.iwi;
  st->iteration_count = W.iteration_count;
  st->pass_last_improver = -1;
  if (!W.has_best) return true;
  size_t off = 0;
  for (int y = 0; y < EG_NY; y++) {
    const std::vector<uint8_t>& run = W.best_actions[y];
    const std::vector<uint8_t>& def = W.best_deficit_actions[y];
    if (off + run.size() + def.size() > EG_UPD_CAT_CAPACITY) return false;
    slot0->len_run[y] = (uint16_t)run.size();
    slot0->len_def[y] = (uint16_t)def.size();
    slot0->off[y] = (uint32_t)off;
    unsigned long long mall = 0ull, mdef = 0ull;
    for (uint8_t a : run) { slot0->cat[off++] = a; mall |= 1ull << a; }
    for (uint8_t a : def) { slot0->cat[off++] = a; mdef |= 1ull << a; }
    slot0->mask_all[y] = mall | mdef;
    slot0->mask_def[y] = mdef;
  }
  return true;
}

void eg_weights_apply_update_state(eg_weights& W, const EgUpdState& st, const EgUpdSlot& slot0, const EgUpdImprovement* improvements,
                                   uint32_t n_improvements, uint32_t iteration0) {
  std::memcpy(W.w, st.w, sizeof(W.w));
  std::memcpy(W.dw, st.dw, sizeof(W.dw));
  W.iwi = st.iwi;
  W.iteration_count = st.iteration_count;
  if (!n_improvements) return;
  Recorded best;  // slot 0 holds the lists of the last improving episode, improvements[n_improvements - 1]
  for (int y = 0; y < EG_NY; y++) {
    const uint8_t* p = slot0.cat + slot0.off[y];
    best.run[y].assign(p, p + slot0.len_run[y]);
    best.deficit[y].assign(p + slot0.len_run[y], p + slot0.len_run[y] + slot0.len_def[y]);
  }
  record_best(W, improvements, n_improvements, iteration0, &st.best_w[0][0], best);
}

EgContrastConsts eg_contrast_consts(const eg_weights& W) {
  EgContrastConsts c;
  c.has_best = W.has_best ? 1 : 0;
  c.force = W.iwi > 800 ? 1 : 0;
  c.best_score = W.has_best ? score_w(W, W.best_metrics) : 0.0;
  c.cost_only = W.optimization_mode == "cost_only" ? 1u : 0u;
  c.threshold = 0.1 * std::max(std::exp(-(double)W.iwi / 500.0), 0.00001 / 0.1);
  c.stagnation = 1.0 + (0.2 * std::pow((double)W.iwi / 10.0, 1.8));
  c.alr = W.learning_rate * (1.0 + 0.1 * (double)W.iwi);
  c.boost = 1.0 + (c.alr * 2.0 * c.stagnation);
  return c;
}

extern "C" {

uint8_t eg_deficit_key_action(uint32_t k) { return (uint8_t)deficit_key_action(k); }

int eg_weights_new(eg_weights** out) {
  if (!out) return eg_fail(EG_ERR_INVALID, "eg_weights_new: out is NULL");
  *out = new eg_weights();
  return EG_OK;
}
void eg_weights_free(eg_weights* w) { delete w; }
int eg_weights_clone(const eg_weights* src, eg_weights** out) {
  if (!src || !out) return eg_fail(EG_ERR_INVALID, "eg_weights_clone: NULL argument");
  *out = new eg_weights(*src);
  return EG_OK;
}

int eg_weights_get_table(const eg_weights* w, eg_weights_table* t) {
  if (!w || !t) return eg_fail(EG_ERR_INVALID, "eg_weights_get_table: NULL argument");
  std::memset(t, 0, sizeof(*t));
  std::memcpy(t->weights, w->w, sizeof(w->w));
  std::memcpy(t->deficit_weights, w->dw, sizeof(w->dw));
  std::memcpy(t->count_weights, w->cw, sizeof(w->cw));
  t->learning_rate = w->learning_rate;
  t->exploration_rate = w->exploration_rate;
  std::memcpy(t->best_metrics, w->best_metrics, sizeof(t->best_metrics));
  t->has_count_weights = w->has_count_weights;
  t->has_best = w->has_best;
  t->iteration_count = w->iteration_count;
  t->iterations_without_improvement = w->iwi;
  return EG_OK;
}
int eg_weights_set_table(eg_weights* w, const eg_weights_table* t) {
  if (!w || !t) return eg_fail(EG_ERR_INVALID, "eg_weights_set_table: NULL argument");
  std::memcpy(w->w, t->weights, sizeof(w->w));
  std::memcpy(w->dw, t->deficit_weights, sizeof(w->dw));
  std::memcpy(w->cw, t->count_weights, sizeof(w->cw));
  w->learning_rate = t->learning_rate;
  w->exploration_rate = t->exploration_rate;
  w->has_count_weights = t->has_count_weights != 0;
  w->iteration_count = t->iteration_count;
  w->iwi = t->iterations_without_improvement;
  return EG_OK;
}
int eg_weights_get_best(const eg_weights* w, uint32_t n_best[EG_N_YEARS], uint8_t* best, size_t best_capacity,
                        uint32_t n_best_deficit[EG_N_YEARS], uint8_t* best_deficit, size_t best_deficit_capacity) {
  if (!w || !n_best || !n_best_deficit) return eg_fail(EG_ERR_INVALID, "eg_weights_get_best: NULL argument");
  size_t ob = 0, obd = 0;
  for (int y = 0; y < EG_NY; y++) {
    n_best[y] = (uint32_t)w->best_actions[y].size();
    n_best_deficit[y] = (uint32_t)w->best_deficit_actions[y].size();
    for (uint8_t a : w->best_actions[y]) {
      if (best && ob < best_capacity) best[ob] = a;
      ob++;
    }
    for (uint8_t a : w->best_deficit_actions[y]) {
      if (best_deficit && obd < best_deficit_capacity) best_deficit[obd] = a;
      obd++;
    }
  }
  return w->has_best ? 1 : 0;
}

int eg_weights_save_json(const eg_weights* w, const char* path) {  // save_to_file, weights/serialization.rs:29-139
  if (!w || !path) return eg_fail(EG_ERR_INVALID, "eg_weights_save_json: NULL argument");
  std::string o = "{\n";
  write_weight_map(o, "weights", &w->w[0][0], EG_N_ACTIONS, false, true);
  o += ",\n  \"learning_rate\": " + egjson::fmt_double(w->learning_rate) + ",\n";
  if (w->has_best) {
    o += "  \"best_metrics\": {\n";
    o += "    \"final_net_emissions\": " + egjson::fmt_double(w->best_metrics[0]) + ",\n";
    o += "    \"average_public_opinion\": " + egjson::fmt_double(w->best_metrics[1]) + ",\n";
    o += "    \"total_cost\": " + egjson::fmt_double(w->best_metrics[2]) + ",\n";
    o += "    \"power_reliability\": " + egjson::fmt_double(w->best_metrics[3]) + "\n  },\n";
  } else {
    o += "  \"best_metrics\": null,\n";
  }
  write_weight_map(o, "best_weights", w->best_weights.data(), EG_N_ACTIONS, false, w->has_best && !w->best_weights.empty());
  o += ",\n";
  write_action_lists(o, "best_actions", w->best_actions, w->has_best);
  o += ",\n  \"iteration_count\": " + std::to_string(w->iteration_count) + ",\n";
  o += "  \"iterations_without_improvement\": " + std::to_string(w->iwi) + ",\n";
  o += "  \"exploration_rate\": " + egjson::fmt_double(w->exploration_rate) + ",\n";
  write_weight_map(o, "deficit_weights", &w->dw[0][0], EG_N_DEFICIT_KEYS, true, true);
  o += ",\n";
  write_action_lists(o, "best_deficit_actions", w->best_deficit_actions, w->has_best);
  o += ",\n  \"optimization_mode\": " + (w->optimization_mode.empty() ? std::string("null") : "\"" + w->optimization_mode + "\"") + ",\n";
  if (w->history.empty()) {
    o += "  \"improvement_history\": null\n";
  } else {
    o += "  \"improvement_history\": [\n";
    for (size_t i = 0; i < w->history.size(); i++) {
      const EgImprovement& h = w->history[i];
      o += "    {\n      \"iteration\": " + std::to_string(h.iteration) + ",\n";
      o += "      \"score\": " + egjson::fmt_double(h.score) + ",\n";
      o += "      \"net_emissions\": " + egjson::fmt_double(h.net_emissions) + ",\n";
      o += "      \"total_cost\": " + egjson::fmt_double(h.total_cost) + ",\n";
      o += "      \"public_opinion\": " + egjson::fmt_double(h.public_opinion) + ",\n";
      o += "      \"power_reliability\": " + egjson::fmt_double(h.power_reliability) + ",\n";
      o += "      \"timestamp\": \"" + h.timestamp + "\"\n    }";
      o += i + 1 < w->history.size() ? ",\n" : "\n";
    }
    o += "  ]\n";
  }
  o += "}";
  std::string tmp = std::string(path) + ".tmp";
  FILE* f = std::fopen(tmp.c_str(), "wb");
  if (!f) return eg_fail(EG_ERR_IO, std::string("cannot write ") + path);
  size_t n = std::fwrite(o.data(), 1, o.size(), f);
  std::fclose(f);
  if (n != o.size() || std::rename(tmp.c_str(), path) != 0) return eg_fail(EG_ERR_IO, std::string("cannot write ") + path);
  return EG_OK;
}

int eg_weights_load_json(const char* path, eg_weights** out) {  // load_from_file, weights/serialization.rs:141-493
  if (!path || !out) return eg_fail(EG_ERR_INVALID, "eg_weights_load_json: NULL argument");
  std::string text;
  if (!egjson::read_file(path, &text)) return eg_fail(EG_ERR_IO, std::string("cannot read ") + path);
  egjson::Value root;
  try {
    root = egjson::Parser(text).parse();
  } catch (const std::exception& ex) {
    return eg_fail(EG_ERR_IO, std::string(path) + ": " + ex.what());
  }
  if (root.kind != egjson::Value::Object || !root.get("weights") || root.get("weights")->kind != egjson::Value::Object)
    return eg_fail(EG_ERR_IO, std::string(path) + ": not a weights file");
  eg_weights* W = new eg_weights();
  if (!read_weight_map(root.get("weights"), &W->w[0][0], EG_N_ACTIONS, false, nullptr)) {
    delete W;
    return eg_fail(EG_ERR_IO, std::string(path) + ": unknown action or generator type, or a year key that is not a u32");
  }
  // deficit weights default to the initial table when the file has none (weights/serialization.rs:266-283)
  if (!read_weight_map(root.get("deficit_weights"), &W->dw[0][0], EG_N_DEFICIT_KEYS, true, nullptr)) {
    delete W;
    return eg_fail(EG_ERR_IO, std::string(path) + ": deficit_weights: a year key that is not a u32");
  }
  if (const egjson::Value* v = root.get("learning_rate")) W->learning_rate = v->num;
  if (const egjson::Value* v = root.get("exploration_rate")) W->exploration_rate = v->num;
  if (!number_as_u32(root.get("iteration_count"), &W->iteration_count) || !number_as_u32(root.get("iterations_without_improvement"), &W->iwi)) {
    delete W;
    return eg_fail(EG_ERR_IO, std::string(path) + ": iteration_count / iterations_without_improvement must be u32");
  }
  if (const egjson::Value* v = root.get("optimization_mode"))
    if (v->kind == egjson::Value::String) W->optimization_mode = v->str;
  const egjson::Value* bm = root.get("best_metrics");
  if (bm && bm->kind == egjson::Value::Object) {
    W->has_best = true;
    if (const egjson::Value* v = bm->get("final_net_emissions")) W->best_metrics[0] = v->num;
    if (const egjson::Value* v = bm->get("average_public_opinion")) W->best_metrics[1] = v->num;
    if (const egjson::Value* v = bm->get("total_cost")) W->best_metrics[2] = v->num;
    if (const egjson::Value* v = bm->get("power_reliability")) W->best_metrics[3] = v->num;
    W->best_weights.assign(&W->w[0][0], &W->w[0][0] + EG_NY * EG_N_ACTIONS);
    // unknown keys are skipped here instead of failing (weights/serialization.rs:286-360)
    const egjson::Value* bw = root.get("best_weights");
    if (bw && bw->kind == egjson::Value::Object)
      for (const auto& kv : bw->obj) {
        int year = std::atoi(kv.first.c_str());
        if (year < EG_BASE_YEAR || year > EG_END_YEAR || kv.second.kind != egjson::Value::Array) continue;
        for (const egjson::Value& entry : kv.second.arr) {
          if (entry.kind != egjson::Value::Array || entry.arr.size() != 2) continue;
          int code = read_action(entry.arr[0]);
          if (code >= 0) W->best_weights[(size_t)(year - EG_BASE_YEAR) * EG_N_ACTIONS + code] = entry.arr[1].num;
        }
      }
    if (!read_action_lists(root.get("best_actions"), W->best_actions) ||
        !read_action_lists(root.get("best_deficit_actions"), W->best_deficit_actions)) {
      delete W;
      return eg_fail(EG_ERR_IO, std::string(path) + ": best actions: a year key that is not a u32");
    }
  }
  const egjson::Value* hist = root.get("improvement_history");
  if (hist && hist->kind == egjson::Value::Array)
    for (const egjson::Value& h : hist->arr) {
      EgImprovement r{};
      number_as_u32(h.get("iteration"), &r.iteration);
      if (const egjson::Value* v = h.get("score")) r.score = v->num;
      if (const egjson::Value* v = h.get("net_emissions")) r.net_emissions = v->num;
      if (const egjson::Value* v = h.get("total_cost")) r.total_cost = v->num;
      if (const egjson::Value* v = h.get("public_opinion")) r.public_opinion = v->num;
      if (const egjson::Value* v = h.get("power_reliability")) r.power_reliability = v->num;
      if (const egjson::Value* v = h.get("timestamp")) r.timestamp = v->str;
      W->history.push_back(r);
    }
  // action_count_weights are not part of the file: empty after load -> heuristic count sampler
  // (weights/serialization.rs:474, sampling.rs:423-442)
  W->has_count_weights = false;
  *out = W;
  return EG_OK;
}

int eg_weights_merge(eg_weights* dst, const eg_weights* other) {  // update_weights_from, strategy.rs:281-311
  if (!dst || !other) return eg_fail(EG_ERR_INVALID, "eg_weights_merge: NULL argument");
  std::memcpy(dst->w, other->w, sizeof(dst->w));
  std::memcpy(dst->dw, other->dw, sizeof(dst->dw));
  if (other->has_count_weights) {
    std::memcpy(dst->cw, other->cw, sizeof(dst->cw));
    dst->has_count_weights = true;
  }
  dst->iteration_count = std::max(dst->iteration_count, other->iteration_count);
  return EG_OK;
}

int eg_update(eg_weights* w, const eg_result* results, const eg_traj* trajs, uint32_t n, uint32_t replay_best,
              uint64_t rng_seed, eg_update_stats* stats_out) {
  if (!w || (n && (!results || !trajs))) return eg_fail(EG_ERR_INVALID, "eg_update: NULL argument");
  eg_update_stats st;
  std::memset(&st, 0, sizeof(st));
  st.n_episodes = n;
  st.batch_best_episode = -1;
  Recorded rec;
  for (uint32_t i = 0; i < n; i++) {
    const double m[4] = {results[i].net_emissions, results[i].public_opinion, results[i].total_cost, results[i].power_reliability};
    rec.from_traj(trajs[i], replay_best != 0);              // transfer_recorded_actions_from
    UpdateRng rng{(uint32_t)rng_seed, (uint32_t)(rng_seed >> 32), w->iteration_count, 0};
    contrast(*w, rec, m, &rng, &st.n_contrast_applied);    // apply_contrast_learning
    if (best_strategy(*w, rec, m)) st.n_improvements++;    // update_best_strategy
    deficit_contrast(*w, rec, &rng);                       // apply_deficit_contrast_learning
    const double sc = score_w(*w, m);
    if (st.batch_best_episode < 0 || sc > st.batch_best_score) { st.batch_best_score = sc; st.batch_best_episode = i; }
    if (results[i].flags) st.n_flagged++;
  }
  st.iterations_without_improvement = w->iwi;
  st.best_score = w->has_best ? score_w(*w, w->best_metrics) : 0.0;
  if (stats_out) *stats_out = st;
  return EG_OK;
}

// Batch-synchronous rule (DESIGN.md §update): the statistics were accumulated against the snapshot `w` (frozen
// best strategy and iterations_without_improvement) by eg_update_stats_device and summed over ranks.
int eg_update_apply_stats(eg_weights* w, const int64_t* stats, uint64_t n_total, const eg_result* best_result,
                          const eg_traj* best_traj, int64_t best_index, eg_update_stats* stats_out) {
  if (!w || !stats) return eg_fail(EG_ERR_INVALID, "eg_update_apply_stats: NULL argument");
  eg_update_stats st;
  std::memset(&st, 0, sizeof(st));
  st.n_episodes = (uint32_t)n_total;
  st.batch_best_episode = best_index;
  const EgContrastConsts c = eg_contrast_consts(*w);
  const int64_t n_pass = stats[1];
  st.n_contrast_applied = (uint32_t)n_pass;
  st.n_flagged = (uint32_t)stats[2];
  if (w->has_best && n_pass > 0) {
    for (int y = 0; y < EG_NY; y++) {
      const int64_t* ys = stats + EG_STATS_HEADER + (size_t)y * EG_STATS_YEAR_STRIDE;
      int occ[EG_N_ACTIONS] = {0};
      for (uint8_t a : w->best_actions[y]) occ[a]++;
      for (uint8_t a : w->best_deficit_actions[y]) occ[a]++;
      for (int k = 0; k < EG_N_ACTIONS; k++) {
        double v = w->w[y][k];
        if (occ[k]) v = std::min(v * std::pow(c.boost, (double)n_pass * (double)occ[k]), kMaxWeight);
        const double lg = ((double)ys[k] + (double)ys[EG_N_ACTIONS + k]) / EG_STATS_FIXED_SCALE;
        if (lg != 0.0) v = std::fmax(v * std::exp(lg), kMinWeight);
        w->w[y][k] = v;
      }
    }
    // randomisation branch of apply_contrast_learning (learning.rs:267-280): the reference perturbs every weight by
    // U(0.75, 1.25) on each iteration once iterations_without_improvement > 1200; the batch rule does it once per batch.
    // The stream is keyed by the iteration count, so every rank draws the same factors.
    if (w->iwi > 1200) {
      UpdateRng rng{0x41424745u, 0x21484354u, w->iteration_count, 0u};
      for (int y = 0; y < EG_NY; y++)
        for (int k = 0; k < EG_N_ACTIONS; k++) w->w[y][k] = egrule::randomise(w->w[y][k], rng.f64());
    }
  }
  // best bookkeeping with the batch winner
  bool improved = false;
  if (best_result && best_traj && n_total > 0) {
    const double m[4] = {best_result->net_emissions, best_result->public_opinion, best_result->total_cost, best_result->power_reliability};
    const double sc = score_w(*w, m);
    st.batch_best_score = sc;
    improved = !w->has_best || sc > score_w(*w, w->best_metrics);
    if (improved) {
      Recorded rec;
      rec.from_traj(*best_traj, false);
      const EgUpdImprovement imp{best_index, sc, {m[0], m[1], m[2], m[3]}};
      record_best(*w, &imp, 1, w->iteration_count, &w->w[0][0], rec);
      st.n_improvements = 1;
    }
  }
  w->iteration_count += (uint32_t)n_total;
  w->iwi = improved ? (uint32_t)(n_total - 1 - (uint64_t)best_index) : w->iwi + (uint32_t)n_total;
  // deficit contrast against the (possibly new) best, with the post-update stagnation counter
  if (w->has_best) {
    const double deterioration = (double)w->iwi / 10.0;
    const double threshold = 0.05 * std::max(std::exp(-(double)w->iwi / 400.0), 0.00001 / 0.05);
    if (deterioration > threshold || w->iwi > 800) {
      const double stagnation = 1.0 + (0.2 * std::pow((double)w->iwi / 10.0, 1.8));
      const double combined = std::pow(deterioration, 0.3) * stagnation;
      const double alr = w->learning_rate * (1.0 + 0.1 * (double)w->iwi);
      const double penalty = 1.0 / (1.0 + alr * 1.5 * combined);
      const double boost = 1.0 + (alr * 2.0 * stagnation * 1.5);
      for (int y = 0; y < EG_NY; y++) {
        const int64_t* hist = stats + EG_STATS_HEADER + (size_t)y * EG_STATS_YEAR_STRIDE + 3 * EG_N_ACTIONS;
        int occ[EG_N_DEFICIT_KEYS] = {0};
        for (uint8_t a : w->best_deficit_actions[y]) {
          int k = deficit_key_of_action(a);
          if (k >= 0) occ[k]++;
        }
        for (int k = 0; k < EG_N_DEFICIT_KEYS; k++) {
          double v = w->dw[y][k];
          if (occ[k]) v = std::min(v * std::pow(boost, (double)n_total * (double)occ[k]), kMaxWeight);
          else if (hist[k] > 0) v = std::fmax(v * std::pow(penalty, (double)hist[k]), kMinWeight);
          w->dw[y][k] = v;
        }
      }
      if (w->iwi > 1200) {  // learning.rs:358-370, once per batch like above
        UpdateRng rng{0x41424745u, 0x44484354u, w->iteration_count, 0u};
        for (int y = 0; y < EG_NY; y++)
          for (int k = 0; k < EG_N_DEFICIT_KEYS; k++) w->dw[y][k] = egrule::randomise(w->dw[y][k], rng.f64());
      }
    }
  }
  st.iterations_without_improvement = w->iwi;
  st.best_score = w->has_best ? score_w(*w, w->best_metrics) : 0.0;
  if (stats_out) *stats_out = st;
  return EG_OK;
}

int eg_weights_history_append(const eg_weights* w, uint64_t iteration, const char* history_path) {
  if (!w || !history_path) return eg_fail(EG_ERR_INVALID, "eg_weights_history_append: NULL argument");
  auto action_display = [](int code) -> std::string {  // impl Display for GridAction, ai/actions/grid_action.rs:18-41
    if (code < 45) return std::string("AddGenerator(") + kGenNames[code / 3] + ", " + std::to_string(kMultPercent[code % 3]) + "%)";
    if (code < 57) return std::string("AddCarbonOffset(") + kOffsetNames[(code - 45) / 3] + ", " + std::to_string(kMultPercent[(code - 45) % 3]) + "%)";
    if (code == EG_ACT_UPGRADE) return "UpgradeEfficiency()";
    if (code == EG_ACT_ADJUST) return "AdjustOperation(, 0%)";
    if (code == EG_ACT_CLOSE) return "CloseGenerator()";
    return "DoNothing";
  };
  const double best_score = w->has_best ? score_w(*w, w->best_metrics) : 0.0;
  char ts[48];
  {
    const std::time_t t = std::time(nullptr);
    std::tm tmv;
    localtime_r(&t, &tmv);
    char tz[8];
    std::strftime(ts, sizeof(ts), "%Y-%m-%dT%H:%M:%S", &tmv);
    std::strftime(tz, sizeof(tz), "%z", &tmv);  // +hhmm -> +hh:mm
    std::string z = tz;
    if (z.size() == 5) z.insert(3, ":");
    std::snprintf(ts + std::strlen(ts), sizeof(ts) - std::strlen(ts), "%s", z.c_str());
  }
  const std::string i2 = "    ", i3 = "      ", i4 = "        ";
  std::string o = "  {\n    \"iteration\": " + std::to_string(iteration) + ",\n    \"timestamp\": \"" + ts + "\",\n    \"weights\": {\n";
  auto rows = [&](const char* name, int n_keys, const double* table, auto key_name, bool present) {
    o += i3 + "\"" + name + "\": {";
    if (present) {
      for (int y = 0; y < EG_NY; y++) {
        o += std::string(y ? "," : "") + "\n" + i4 + "\"" + std::to_string(EG_BASE_YEAR + y) + "\": {";
        for (int k = 0; k < n_keys; k++)
          o += std::string(k ? "," : "") + "\n" + i4 + "  \"" + key_name(k) + "\": " + egjson::fmt_double(table[(size_t)y * n_keys + k]);
        o += "\n" + i4 + "}";
      }
      o += "\n" + i3;
    }
    o += "}";
  };
  rows("weights", EG_N_ACTIONS, &w->w[0][0], [&](int k) { return action_display(k); }, true);
  o += ",\n";
  rows("action_count_weights", EG_N_COUNT_KEYS, &w->cw[0][0], [&](int k) { return std::to_string(k); }, w->has_count_weights);
  o += ",\n" + i3 + "\"learning_rate\": " + egjson::fmt_double(w->learning_rate);
  o += ",\n" + i3 + "\"iteration_count\": " + std::to_string(w->iteration_count);
  o += ",\n" + i3 + "\"iterations_without_improvement\": " + std::to_string(w->iwi);
  o += ",\n" + i3 + "\"exploration_rate\": " + egjson::fmt_double(w->exploration_rate);
  o += ",\n" + i3 + "\"force_best_actions\": false";
  o += ",\n";
  rows("deficit_weights", EG_N_DEFICIT_KEYS, &w->dw[0][0], [&](int k) { return action_display(deficit_key_action(k)); }, true);
  o += ",\n" + i3 + "\"guaranteed_best_actions\": false";
  o += ",\n" + i3 + "\"optimization_mode\": " + (w->optimization_mode.empty() ? std::string("null") : "\"" + w->optimization_mode + "\"");
  o += ",\n" + i3 + "\"best_score\": " + egjson::fmt_double(best_score) + "\n" + i2 + "},\n";
  o += i2 + "\"best_score\": " + egjson::fmt_double(best_score) + "\n  }";
  // append to the array without re-parsing it: the file is only ever written by this function (or is "[]" / missing)
  std::string text;
  egjson::read_file(history_path, &text);
  size_t end = text.find_last_of(']');
  std::string head = end == std::string::npos ? "[" : text.substr(0, end);
  while (!head.empty() && (head.back() == ' ' || head.back() == '\n' || head.back() == '\t' || head.back() == '\r')) head.pop_back();
  const bool first = head.empty() || head == "[";
  if (head.empty()) head = "[";
  const std::string out = head + (first ? "\n" : ",\n") + o + "\n]";
  std::FILE* f = std::fopen(history_path, "w");
  if (!f) return eg_fail(EG_ERR_IO, std::string("cannot write ") + history_path);
  std::fwrite(out.data(), 1, out.size(), f);
  std::fclose(f);
  return EG_OK;
}

int eg_update_combine_apply(eg_weights* w, const int64_t* stats_sum, const void* records, uint32_t n_records, uint64_t n_total,
                            uint64_t first_episode, eg_update_stats* stats_out) {
  if (!w || !stats_sum || (!records && n_records)) return eg_fail(EG_ERR_INVALID, "eg_update_combine_apply: NULL argument");
  const unsigned char* rec = (const unsigned char*)records;
  const unsigned char* win = nullptr;
  double win_score = 0.0;
  int64_t win_id = 0;
  for (uint32_t r = 0; r < n_records; r++) {
    const unsigned char* p = rec + (size_t)r * EG_BEST_RECORD_BYTES;
    double score;
    int64_t id;
    std::memcpy(&score, p, 8);
    std::memcpy(&id, p + 8, 8);
    if (!win || score > win_score || (score == win_score && id < win_id)) { win = p; win_score = score; win_id = id; }
  }
  if (!win) return eg_update_apply_stats(w, stats_sum, n_total, nullptr, nullptr, -1, stats_out);
  if (n_total > 0 && (win_id < (int64_t)first_episode || (uint64_t)(win_id - (int64_t)first_episode) >= n_total))
    return eg_fail(EG_ERR_INVALID, "eg_update_combine_apply: the winner record's episode id lies outside the batch");
  eg_result res;
  eg_traj traj;
  std::memcpy(&res, win + 16, sizeof(res));
  std::memcpy(&traj, win + 16 + sizeof(res), sizeof(traj));
  return eg_update_apply_stats(w, stats_sum, n_total, &res, &traj, win_id - (int64_t)first_episode, stats_out);
}

}  // extern "C"
