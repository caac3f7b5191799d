// eirgrid_host.cpp — native host driver of the B200 episode engine: the reference's aiSimulator command line
// (aiSimulator/src/cli/cli.rs:3-59, src/main.rs:31-193) and batch/checkpoint loop (src/core/multi_simulation.rs:95-611)
// on top of the C ABI in include/eirgrid_b200.h. The reference host is Rust; no Rust toolchain exists in this image, so the
// host is C++17 (INTEGRATION.md has the Rust shim). Nothing here touches CUDA directly: every device operation is a call
// into libeirgrid_b200.so.
//
//   eirgrid_host -n 1000000 --assets aiSimulator/assets --no-continue [--devices 0,1,2,3] [--batch-size 65536]
//
// One process drives 1..8 GPUs: per batch every GPU rolls out its shard of episode ids (eg_train_batch_begin is
// asynchronous), the per-GPU statistics tables are summed on the host (5,156 int64 words each — the single-process form
// of the allreduce the one-process-per-GPU Python driver does with NCCL) and the identical update is applied once.
#include <dirent.h>
#include <sys/stat.h>
#include <sys/types.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <string>
#include <vector>

#include "../include/eirgrid_b200.h"

namespace {

constexpr int kFullRunPercentage = 10;              // multi_simulation.rs:38
constexpr bool kReplayBestStrategyInFullRuns = true;  // multi_simulation.rs:39

struct Args {  // cli/cli.rs:3-59, same names and defaults
  uint64_t iterations = 1000;
  bool parallel = true;
  bool no_continue = false;
  std::string checkpoint_dir = "checkpoints";
  uint64_t checkpoint_interval = 5;
  uint64_t progress_interval = 10;
  std::string cache_dir = "cache";
  bool force_full_simulation = false;
  bool enable_timing = false;
  bool has_seed = false;
  uint64_t seed = 0;
  bool verbose_state_logging = false;
  bool cost_only = false;
  bool enable_energy_sales = true;
  bool enable_csv_export = true;
  bool debug_logging = false;
  bool debug_weights = false;
  bool enable_construction_delays = false;
  bool track_weight_history = false;
  // additions of this implementation
  std::string assets = "aiSimulator/assets";
  uint32_t batch_size = 65536;
  std::string update_mode = "batch";
  bool has_master_seed = false;
  uint64_t master_seed = 0;
  std::vector<int> devices = {0};
};

[[noreturn]] void die(const std::string& msg) {
  std::fprintf(stderr, "error: %s\n", msg.c_str());
  std::exit(2);
}

void check(int rc, const char* what) {
  if (rc < 0) die(std::string(what) + ": " + eg_last_error());
}

void usage() {
  std::puts(
      "EirGrid Power System Simulator (2025-2050), B200 episode engine\n\n"
      "  -n, --iterations <N>            Number of simulation iterations [default: 1000]\n"
      "  -p, --parallel                  Run simulations in parallel (always on)\n"
      "      --no-continue               Start fresh instead of continuing from the newest checkpoint\n"
      "  -c, --checkpoint-dir <DIR>      [default: checkpoints]\n"
      "  -i, --checkpoint-interval <N>   [default: 5]\n"
      "  -r, --progress-interval <S>     [default: 10]\n"
      "  -C, --cache-dir <DIR>           [default: cache]\n"
      "      --force-full-simulation\n"
      "      --enable-timing\n"
      "      --seed <SEED>               Random seed for deterministic simulation (every episode re-seeded with it)\n"
      "  -v, --verbose-state-logging\n"
      "      --cost-only                 Optimize for cost only\n"
      "      --enable-energy-sales       (always on)\n"
      "      --enable-csv-export         (always on: summary, improvement history and settlements CSVs of the best run)\n"
      "      --debug-logging, --debug-weights, --track-weight-history\n"
      "      --enable-construction-delays\n"
      "additions: --assets <DIR> --batch-size <N> --update-mode batch|sequential --master-seed <S> --devices 0,1,..");
}

Args parse(int argc, char** argv) {
  Args a;
  auto need = [&](int& i) -> std::string {
    if (i + 1 >= argc) die(std::string("missing value for ") + argv[i]);
    return argv[++i];
  };
  // unsigned decimal integers only (clap's usize/u64 parser): no sign, no garbage, no overflow
  auto number = [&](int& i, uint64_t max) -> uint64_t {
    const std::string flag = argv[i], v = need(i);
    uint64_t x = 0;
    bool ok = !v.empty() && v.size() <= 20;
    for (char ch : v) {
      if (ch < '0' || ch > '9' || x > (UINT64_MAX - (uint64_t)(ch - '0')) / 10) { ok = false; break; }
      x = x * 10 + (uint64_t)(ch - '0');
    }
    if (!ok || x > max) die("invalid value '" + v + "' for '" + flag + "'");
    return x;
  };
  for (int i = 1; i < argc; i++) {
    const std::string f = argv[i];
    if (f == "-n" || f == "--iterations") a.iterations = number(i, UINT64_MAX);
    else if (f == "-p" || f == "--parallel") a.parallel = true;
    else if (f == "--no-continue") a.no_continue = true;
    else if (f == "-c" || f == "--checkpoint-dir") a.checkpoint_dir = need(i);
    else if (f == "-i" || f == "--checkpoint-interval") a.checkpoint_interval = std::max<uint64_t>(1, number(i, UINT64_MAX));
    else if (f == "-r" || f == "--progress-interval") a.progress_interval = number(i, UINT64_MAX);
    else if (f == "-C" || f == "--cache-dir") a.cache_dir = need(i);
    else if (f == "--force-full-simulation") a.force_full_simulation = true;
    else if (f == "--enable-timing") a.enable_timing = true;
    else if (f == "--seed") { a.has_seed = true; a.seed = number(i, UINT64_MAX); }
    else if (f == "-v" || f == "--verbose-state-logging") a.verbose_state_logging = true;
    else if (f == "--cost-only") a.cost_only = true;
    else if (f == "--enable-energy-sales") a.enable_energy_sales = true;
    else if (f == "--enable-csv-export") a.enable_csv_export = true;
    else if (f == "--debug-logging") a.debug_logging = true;
    else if (f == "--debug-weights") a.debug_weights = true;
    else if (f == "--enable-construction-delays") a.enable_construction_delays = true;
    else if (f == "--track-weight-history") a.track_weight_history = true;
    else if (f == "--assets") a.assets = need(i);
    else if (f == "--batch-size") a.batch_size = (uint32_t)number(i, UINT32_MAX);
    else if (f == "--update-mode") a.update_mode = need(i);
    else if (f == "--master-seed") { a.has_master_seed = true; a.master_seed = number(i, UINT64_MAX); }
    else if (f == "--devices") {
      a.devices.clear();
      std::string v = need(i), cur;
      for (char ch : v + ",") {
        if (ch == ',') { if (!cur.empty()) a.devices.push_back(std::stoi(cur)); cur.clear(); }
        else if (ch < '0' || ch > '9' || cur.size() >= 4) die("invalid value '" + v + "' for '--devices'");
        else cur += ch;
      }
      if (a.devices.empty()) die("--devices needs at least one index");
    } else if (f == "-h" || f == "--help") { usage(); std::exit(0); }
    else die("unknown argument " + f);
  }
  if (a.update_mode != "batch" && a.update_mode != "sequential") die("--update-mode must be batch or sequential");
  if (a.update_mode != "batch" && a.devices.size() > 1) die("--update-mode sequential is single-GPU");
  if (a.batch_size == 0) die("--batch-size must be positive");
  return a;
}

bool is_dir(const std::string& p) {
  struct stat st;
  return stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}
bool exists(const std::string& p) {
  struct stat st;
  return stat(p.c_str(), &st) == 0;
}
void mkdirs(const std::string& p) {
  std::string cur;
  for (size_t i = 0; i <= p.size(); i++) {
    if (i == p.size() || p[i] == '/') {
      if (!cur.empty() && !is_dir(cur) && mkdir(cur.c_str(), 0777) != 0 && !is_dir(cur)) die("cannot create directory " + cur);
    }
    if (i < p.size()) cur += p[i];
  }
}
std::vector<std::string> list_dir(const std::string& p) {
  std::vector<std::string> out;
  if (DIR* d = opendir(p.c_str())) {
    while (dirent* e = readdir(d)) {
      const std::string n = e->d_name;
      if (n != "." && n != "..") out.push_back(n);
    }
    closedir(d);
  }
  std::sort(out.begin(), out.end());
  return out;
}

// "2024" + %m%d_%H%M%S: the literal prefix is the reference's (multi_simulation.rs:161-163)
std::string run_dir_name() {
  const std::time_t t = std::time(nullptr);
  std::tm tmv;
  localtime_r(&t, &tmv);
  char buf[32];
  std::strftime(buf, sizeof(buf), "%m%d_%H%M%S", &tmv);
  return std::string("2024") + buf;
}

bool digits_or_underscore(const std::string& n) {
  return !n.empty() && std::all_of(n.begin(), n.end(), [](char c) { return (c >= '0' && c <= '9') || c == '_'; });
}
// multi_simulation.rs:219-234
bool valid_run_dir(const std::string& n) {
  if (n.size() != 15 || !digits_or_underscore(n)) return false;
  for (int i = 0; i < 8; i++)
    if (n[i] < '0' || n[i] > '9') return false;
  const int year = std::stoi(n.substr(0, 4)), month = std::stoi(n.substr(4, 2)), day = std::stoi(n.substr(6, 2));
  return !(year > 2025 || month > 12 || day > 31);
}

// newest directory the reference would resume from ("" if none)
std::string find_resume_dir(const std::string& checkpoint_dir) {
  std::string best;
  for (const std::string& n : list_dir(checkpoint_dir))
    if (is_dir(checkpoint_dir + "/" + n) && valid_run_dir(n) && n > best) best = n;
  return best.empty() ? "" : checkpoint_dir + "/" + best;
}

// multi_simulation.rs:385-413
uint64_t find_start_iteration(const std::string& checkpoint_dir) {
  std::string best;
  for (const std::string& n : list_dir(checkpoint_dir))
    if (is_dir(checkpoint_dir + "/" + n) && digits_or_underscore(n) && n > best) best = n;
  if (best.empty()) return 0;
  std::ifstream f(checkpoint_dir + "/" + best + "/checkpoint_iteration.txt");
  uint64_t v = 0;
  if (!(f >> v)) return 0;
  return v;
}

// latest_weights.json overlaid with every thread_*_weights.json (multi_simulation.rs:237-290)
eg_weights* load_initial_weights(const Args& a) {
  eg_weights* fresh = nullptr;
  check(eg_weights_new(&fresh), "eg_weights_new");
  if (a.no_continue) {
    std::puts("Starting fresh simulation (--no-continue specified)");
    return fresh;
  }
  const std::string latest = find_resume_dir(a.checkpoint_dir);
  if (latest.empty()) {
    std::puts("No checkpoint directories found, starting fresh");
    return fresh;
  }
  eg_weights* merged = nullptr;
  bool found = false;
  if (eg_weights_load_json((latest + "/latest_weights.json").c_str(), &merged) == 0) found = true;
  else check(eg_weights_new(&merged), "eg_weights_new");
  for (const std::string& n : list_dir(latest)) {
    if (n.rfind("thread_", 0) != 0 || n.size() < 20 || n.substr(n.size() - 13) != "_weights.json") continue;
    eg_weights* t = nullptr;
    if (eg_weights_load_json((latest + "/" + n).c_str(), &t) == 0) {
      check(eg_weights_merge(merged, t), "eg_weights_merge");
      eg_weights_free(t);
      found = true;
    }
  }
  if (!found) {
    std::puts("No weights found in latest directory, starting fresh");
    eg_weights_free(merged);
    return fresh;
  }
  std::printf("Loaded weights from %s\n", latest.c_str());
  eg_weights_free(fresh);
  return merged;
}

double best_score_of(const eg_weights* w, bool* has_best) {
  eg_weights_table t;
  check(eg_weights_get_table(w, &t), "eg_weights_get_table");
  *has_best = t.has_best != 0;
  if (!t.has_best) return 0.0;
  const double net = t.best_metrics[0], opinion = t.best_metrics[1], cost = t.best_metrics[2];
  if (net > 0.0) return 1.0 - std::min(net / 1000000.0, 1.0);  // scoring.rs:18-44
  const double normalized = std::max(cost / 50000000000.0, 1.0);
  const double cs = 1.0 - std::min(std::log(normalized) / std::log(100.0), 1.0);
  const double cw = normalized > 8.0 ? 0.8 : 0.5;
  return 1.0 + (cs * cw + opinion * (1.0 - cw));
}

double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace

int main(int argc, char** argv) {
  const Args a = parse(argc, argv);
  std::puts("EirGrid Power System Simulator (2025-2050)");
  const size_t G = a.devices.size();
  std::vector<eg_ctx*> ctx(G, nullptr);
  const std::string sj = a.assets + "/settlements.json", gc = a.assets + "/ireland_generators.csv", cj = a.assets + "/coastline_points.json";
  for (size_t g = 0; g < G; g++) {
    check(eg_init(a.devices[g], nullptr, &ctx[g]), "eg_init");
    check(eg_map_load(ctx[g], sj.c_str(), gc.c_str(), cj.c_str()), "eg_map_load");
  }
  uint32_t info[4];
  check(eg_map_info(ctx[0], info), "eg_map_info");
  std::printf("Map: %u settlements, %u existing generators, %u coastline points, %u x %u candidate sites, %zu GPU(s)\n", info[0], info[1],
              info[2], info[3], info[3], G);

  mkdirs(a.checkpoint_dir);
  eg_weights* weights = load_initial_weights(a);
  const uint64_t start_iteration = a.no_continue ? 0 : find_start_iteration(a.checkpoint_dir);
  const std::string run_dir = a.checkpoint_dir + "/" + run_dir_name();
  mkdirs(run_dir);
  const bool cache_loaded = exists(a.cache_dir + "/location_analysis.json");  // load_location_analysis, multi_simulation.rs:149-154
  if (!cache_loaded) std::printf("Warning: Location analysis cache not found in %s. All simulations will use full mode.\n", a.cache_dir.c_str());
  const bool same_stream = a.has_seed;  // --seed re-seeds every episode with the same value (simulation.rs:50-52)
  const uint64_t rng_seed = a.has_seed ? a.seed : (a.has_master_seed ? a.master_seed : (uint64_t)std::time(nullptr) * 2654435761ull);
  const uint64_t remaining0 = a.iterations > start_iteration ? a.iterations - start_iteration : 0;
  const uint32_t per_gpu = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(a.batch_size, (std::max<uint64_t>(remaining0, 1) + G - 1) / G));
  const uint64_t final_full = a.iterations * kFullRunPercentage / 100;
  std::printf("Starting multi-simulation optimization with %llu iterations (%llu completed, %llu remaining) in directory %s\n",
              (unsigned long long)a.iterations, (unsigned long long)start_iteration, (unsigned long long)remaining0, run_dir.c_str());

  std::vector<int64_t> stats(EG_STATS_WORDS), shard_stats(EG_STATS_WORDS);
  std::vector<unsigned char> records(G * EG_BEST_RECORD_BYTES);
  uint64_t completed = start_iteration;
  uint64_t next_checkpoint = (completed / a.checkpoint_interval + 1) * a.checkpoint_interval;
  const double t_start = now_s();
  double t_progress = t_start;
  eg_update_stats st{};
  uint64_t n_flagged = 0;
  double t_train = 0.0;        // wall time of the training batches (device statistics path)
  uint64_t n_train = 0;
  double t_inorder = 0.0;      // wall time of the batches under the per-episode rule (replay phase, sequential modes)
  uint64_t n_inorder = 0;
  while (completed < a.iterations) {
    const double t_batch = now_s();
    const bool is_full_run = a.force_full_simulation || !cache_loaded || completed + final_full >= a.iterations;
    uint32_t nb[EG_N_YEARS], nbd[EG_N_YEARS];
    const bool has_best_actions = eg_weights_get_best(weights, nb, nullptr, 0, nbd, nullptr, 0) == 1;
    eg_run_cfg cfg{};
    cfg.cost_only = a.cost_only;
    cfg.enable_energy_sales = a.enable_energy_sales;
    cfg.enable_construction_delays = a.enable_construction_delays;
    cfg.replay_best = is_full_run && kReplayBestStrategyInFullRuns && has_best_actions;
    cfg.same_stream_all_episodes = same_stream;
    uint64_t done_now = 0;
    if (a.update_mode == "batch" && !cfg.replay_best) {
      // never past the requested iteration count, nor past the start of the replay phase: the last batch is smaller, and
      // ragged over the GPUs (the first `rem` devices take one episode more)
      const uint64_t phase_end = (is_full_run || final_full >= a.iterations) ? a.iterations : a.iterations - final_full;
      done_now = std::min<uint64_t>((uint64_t)per_gpu * G, phase_end - completed);
      const uint64_t base = done_now / G, rem = done_now % G;
      for (size_t g = 0; g < G; g++)
        check(eg_train_batch_begin(ctx[g], weights, &cfg, rng_seed, completed + g * base + std::min<uint64_t>(g, rem), (uint32_t)(base + (g < rem ? 1 : 0))),
              "eg_train_batch_begin");
      std::fill(stats.begin(), stats.end(), 0);
      for (size_t g = 0; g < G; g++) {
        check(eg_train_batch_end(ctx[g], shard_stats.data(), records.data() + g * EG_BEST_RECORD_BYTES), "eg_train_batch_end");
        for (size_t i = 0; i < stats.size(); i++) stats[i] += shard_stats[i];
      }
      check(eg_update_combine_apply(weights, stats.data(), records.data(), (uint32_t)G, done_now, completed, &st), "eg_update_combine_apply");
      t_train += now_s() - t_batch;
      n_train += done_now;
    } else {
      // replay batches and --update-mode sequential: the reference's per-episode update in episode order on the GPU
      // (eg_update_device behind eg_train_batch_inorder; it rebuilds the doubled records of replay iterations, quirk Q10)
      const uint64_t phase_end = (is_full_run || final_full >= a.iterations) ? a.iterations : a.iterations - final_full;
      const uint32_t n_s = (uint32_t)std::min<uint64_t>(per_gpu, phase_end - completed);
      check(eg_train_batch_inorder(ctx[0], weights, &cfg, rng_seed, completed, n_s, rng_seed, &st), "eg_train_batch_inorder");
      done_now = n_s;
      t_inorder += now_s() - t_batch;
      n_inorder += done_now;
    }
    completed += done_now;
    if (st.n_flagged) {
      n_flagged += st.n_flagged;
      std::fprintf(stderr, "warning: %u episodes of this batch carry eg_result.flags (replay-phase years with more than 40 recorded actions, quirk Q10; or a capacity overflow)\n", st.n_flagged);
    }
    const double t = now_s();
    if (t - t_progress >= (double)a.progress_interval) {
      t_progress = t;
      std::printf("Progress: %llu/%llu iterations, %.0f iterations/s, best score %.6f, %u without improvement\n", (unsigned long long)completed,
                  (unsigned long long)a.iterations, (double)(completed - start_iteration) / std::max(t - t_start, 1e-9), st.best_score,
                  st.iterations_without_improvement);
    }
    if (completed >= next_checkpoint || completed >= a.iterations) {  // multi_simulation.rs:544-567
      next_checkpoint = (completed / a.checkpoint_interval + 1) * a.checkpoint_interval;
      check(eg_weights_save_json(weights, (run_dir + "/latest_weights.json").c_str()), "eg_weights_save_json");
      std::ofstream(run_dir + "/checkpoint_iteration.txt") << std::min(completed, a.iterations);
      if (a.track_weight_history)
        check(eg_weights_history_append(weights, completed, (run_dir + "/weight_history.json").c_str()), "eg_weights_history_append");
    }
  }
  const double elapsed = now_s() - t_start;
  check(eg_weights_save_json(weights, (run_dir + "/best_weights.json").c_str()), "eg_weights_save_json");  // multi_simulation.rs:1161-1163
  bool has_best = false;
  const double best = best_score_of(weights, &has_best);
  if (a.enable_csv_export && has_best) {  // multi_simulation.rs:852-925: <run_dir>/enhanced_csv/<timestamp>/
    eg_run_cfg cfg{};
    cfg.cost_only = a.cost_only;
    cfg.enable_energy_sales = a.enable_energy_sales;
    char written[512];
    check(eg_export_best_run_csv(ctx[0], weights, &cfg, (run_dir + "/enhanced_csv").c_str(), written), "eg_export_best_run_csv");
    std::printf("Enhanced simulation results exported to: %s\n", written);
  }
  uint64_t launches = 0;
  for (size_t g = 0; g < G; g++) launches += eg_kernel_launches(ctx[g]);
  std::printf("{\"run_dir\": \"%s\", \"iterations\": %llu, \"start_iteration\": %llu, \"elapsed_s\": %.3f, \"episodes_per_s\": %.1f, "
              "\"training_batches\": {\"episodes\": %llu, \"episodes_per_s\": %.1f}, \"per_episode_rule_batches\": {\"episodes\": %llu, \"seconds\": %.3f}, "
              "\"best_score\": %s, \"iterations_without_improvement\": %u, \"flagged_episodes\": %llu, \"n_gpus\": %zu, \"kernel_launches\": %llu}\n",
              run_dir.c_str(), (unsigned long long)completed, (unsigned long long)start_iteration, elapsed,
              (double)(completed - start_iteration) / std::max(elapsed, 1e-9), (unsigned long long)n_train, (double)n_train / std::max(t_train, 1e-9),
              (unsigned long long)n_inorder, t_inorder,
              has_best ? std::to_string(best).c_str() : "null",
              st.iterations_without_improvement, (unsigned long long)n_flagged, G, (unsigned long long)launches);
  eg_weights_free(weights);
  for (eg_ctx* c : ctx) eg_destroy(c);
  return 0;
}
