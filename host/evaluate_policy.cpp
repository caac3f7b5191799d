// evaluate_policy — statistics of a policy table over many episodes on one or more GPUs, through the C ABI only.
//
//   evaluate_policy --weights best_weights.json --assets aiSimulator/assets -n 1048576 [--seed S] [--first-episode K]
//                   [--cost-only] [--no-yearly] [--json OUT] [--devices 0,1,..]
//
// The flags of `python -m eirgrid_b200.evaluate`, plus --devices. Each device takes a contiguous share of the episode ids (total /
// devices each, the first total % devices one more, like trainer.shard_of) and is driven by its own host thread with its own
// context; the shards' records are merged in device order with eg_eval_stats_merge, so the result does not depend on which
// thread finishes first, and the JSON is written by eg_eval_stats_write_json (to stdout without --json).
#include <unistd.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../include/eirgrid_b200.h"

namespace {

[[noreturn]] void usage_error(const std::string& msg) {
  std::fprintf(stderr, "error: %s\n", msg.c_str());
  std::exit(2);
}

struct Shard {
  int device = 0;
  uint64_t first = 0, n = 0;
  eg_eval_stats stats;
  int rc = 0;
  std::string error;
};

void run_shard(Shard* s, const std::string& weights, const std::string& assets, const eg_run_cfg& cfg, uint64_t seed, uint32_t yearly) {
  eg_ctx* ctx = nullptr;
  eg_weights* w = nullptr;
  std::memset(&s->stats, 0, sizeof(s->stats));
  const char* step = "eg_init";
  s->rc = eg_init(s->device, nullptr, &ctx);
  if (s->rc >= 0) {
    step = "eg_map_load";
    s->rc = eg_map_load(ctx, (assets + "/settlements.json").c_str(), (assets + "/ireland_generators.csv").c_str(),
                        (assets + "/coastline_points.json").c_str());
  }
  if (s->rc >= 0) { step = "eg_weights_load_json"; s->rc = eg_weights_load_json(weights.c_str(), &w); }
  if (s->rc >= 0) { step = "eg_evaluate"; s->rc = eg_evaluate(ctx, w, &cfg, seed, s->first, s->n, yearly, &s->stats); }
  if (s->rc < 0) s->error = std::string(step) + " on device " + std::to_string(s->device) + ": " + eg_last_error();
  if (w) eg_weights_free(w);
  if (ctx) eg_destroy(ctx);
}

}  // namespace

int main(int argc, char** argv) {
  std::string weights, assets, json;
  uint64_t n = 0, seed = 1, first_episode = 0;
  bool has_n = false, cost_only = false, no_yearly = false;
  std::vector<int> devices = {0};
  auto need = [&](int& i) -> std::string {
    if (i + 1 >= argc) usage_error(std::string("missing value for ") + argv[i]);
    return argv[++i];
  };
  auto number = [&](int& i) -> uint64_t {  // unsigned decimal integers only: no sign, no garbage, no overflow
    const std::string flag = argv[i], v = need(i);
    uint64_t x = 0;
    bool ok = !v.empty();
    for (char ch : v) {
      if (ch < '0' || ch > '9' || x > (UINT64_MAX - (uint64_t)(ch - '0')) / 10) { ok = false; break; }
      x = x * 10 + (uint64_t)(ch - '0');
    }
    if (!ok) usage_error("invalid value '" + v + "' for '" + flag + "'");
    return x;
  };
  for (int i = 1; i < argc; i++) {
    const std::string f = argv[i];
    if (f == "--weights") weights = need(i);
    else if (f == "--assets") assets = need(i);
    else if (f == "-n" || f == "--episodes") { n = number(i); has_n = true; }
    else if (f == "--seed") seed = number(i);
    else if (f == "--first-episode") first_episode = number(i);
    else if (f == "--cost-only") cost_only = true;
    else if (f == "--no-yearly") no_yearly = true;
    else if (f == "--json") json = need(i);
    else if (f == "--devices") {
      devices.clear();
      const std::string v = need(i);
      std::string cur;
      for (char ch : v + ",") {
        if (ch == ',') { if (!cur.empty()) devices.push_back(std::atoi(cur.c_str())); cur.clear(); }
        else if (ch < '0' || ch > '9' || cur.size() >= 4) usage_error("invalid value '" + v + "' for '--devices'");
        else cur += ch;
      }
      if (devices.empty()) usage_error("--devices needs at least one index");
    } else if (f == "-h" || f == "--help") {
      std::puts("evaluate_policy --weights <PATH> --assets <DIR> -n <N> [--seed <S=1>] [--first-episode <K=0>] [--cost-only] [--no-yearly]\n"
                "                [--json <OUT>] [--devices 0,1,..]");
      return 0;
    } else usage_error("unknown argument " + f);
  }
  if (weights.empty() || assets.empty() || !has_n) usage_error("--weights, --assets and -n are required");

  eg_run_cfg cfg;
  std::memset(&cfg, 0, sizeof(cfg));
  cfg.cost_only = cost_only ? 1u : 0u;
  cfg.enable_energy_sales = 1;
  const uint64_t world = devices.size(), base = n / world, rem = n % world;
  std::vector<Shard> shards(world);
  std::vector<std::thread> threads;
  for (uint64_t r = 0; r < world; r++) {
    shards[r].device = devices[r];
    shards[r].first = first_episode + r * base + (r < rem ? r : rem);
    shards[r].n = base + (r < rem ? 1 : 0);
    threads.emplace_back(run_shard, &shards[r], weights, assets, cfg, seed, no_yearly ? 0u : 1u);
  }
  for (std::thread& t : threads) t.join();
  eg_eval_stats total;
  std::memset(&total, 0, sizeof(total));
  for (const Shard& s : shards) {
    if (s.rc < 0) {
      std::fprintf(stderr, "error: %s\n", s.error.c_str());
      return 1;
    }
    if (eg_eval_stats_merge(&total, &s.stats) < 0) {
      std::fprintf(stderr, "error: eg_eval_stats_merge: %s\n", eg_last_error());
      return 1;
    }
  }
  std::string path = json;
  char tmp[] = "/tmp/evaluate_policy_XXXXXX";
  if (path.empty()) {
    const int fd = mkstemp(tmp);
    if (fd < 0) { std::fprintf(stderr, "error: cannot create a temporary file\n"); return 1; }
    close(fd);
    path = tmp;
  }
  const int rc = eg_eval_stats_write_json(&total, path.c_str());
  if (rc >= 0 && json.empty()) {
    if (std::FILE* f = std::fopen(path.c_str(), "rb")) {
      char buf[65536];
      size_t k;
      while ((k = std::fread(buf, 1, sizeof(buf), f)) > 0) std::fwrite(buf, 1, k, stdout);
      std::fclose(f);
    }
  }
  if (json.empty()) std::remove(tmp);
  if (rc < 0) {
    std::fprintf(stderr, "error: eg_eval_stats_write_json: %s\n", eg_last_error());
    return 1;
  }
  return 0;
}
