// engine.cu — device context and the C-ABI entry points of include/eirgrid_b200.h.
// There is no CPU fallback: every compute entry point needs a CUDA device and fails with
// EG_ERR_NO_DEVICE / EG_ERR_CUDA otherwise.
#include <cuda_runtime.h>
#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include "common.hpp"
#include "device_buffer.hpp"
#include "episode.cuh"
#include "host_tables.hpp"
#include "site_tables.cuh"
#include "stats.cuh"
#include "suitability.cuh"
#include "update.cuh"
#include "weights.hpp"

static_assert(sizeof(EgPolicyDevice) == 38784, "bench.py and eirgrid_b200/_abi.py quote this size");
static thread_local std::string g_last_error;
int eg_fail(int code, const std::string& message) {
  g_last_error = message;
  return code;
}

#define EG_CUDA(expr)                                                                                   \
  do {                                                                                                  \
    cudaError_t err__ = (expr);                                                                         \
    if (err__ != cudaSuccess)                                                                           \
      return eg_fail(EG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(err__));               \
  } while (0)

struct eg_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  OwnedStream own_stream;              // set when eg_init created the stream; a stream passed in stays the caller's
  uint64_t launches = 0;
  bool map_ready = false;
  bool policy_ready = false;
  bool policy_count_weights = false;
  bool policy_stagnation = false;
  EgHostMap hmap;
  EgHostTables htab;
  EgDeviceMap dmap{};
  // Device memory in groups that live equally long, each allocated all or nothing: built in a local and moved in only when
  // every allocation succeeded, so a failed call leaves the group absent and the next call allocates it again.
  struct MapTables {  // the loaded map (build_device_map)
    DeviceArray<EgSmallTables> small;
    DeviceArray<double> plant_terms, near, sx, sy, ex, ey, cx, cy, site_opinion, coast;
    DeviceArray<double> prefix, walk;  // [6][26][ns], [7][26][ns][2]
    DeviceArray<uint16_t> order;       // [7][26][ns]
    DeviceArray<int> r2_limit;
    DeviceArray<uint32_t> pop;
    DeviceArray<double> urban_r;       // [26][S] sqrt(pop) * 5 (is_urban_area, map_handler.rs:1199-1209)
    double urban_r_max = 0.0;
  } map;
  struct PolicyBuffers {  // the weights snapshot the rollouts read
    DeviceArray<EgPolicyDevice> d;
    PinnedArray<EgPolicyDevice> h[2];  // pinned staging of the snapshot, used in turn
    Event copied[2];                   // the H2D copy issued from h[b] has completed
  } policy;
  int policy_turn = 0;
  struct Scratch {  // outputs of the host-buffer entry points, each grown on demand
    DeviceArray<eg_result> out;
    DeviceArray<eg_traj> traj, traj_in;
    DeviceArray<eg_sites> sites;
    DeviceArray<eg_yearly> yearly;
  } scratch;
  struct TrainBuffers {  // eg_train_batch_*: statistics table, shard best, winner record (device) and their pinned host mirrors
    DeviceArray<int64_t> stats;
    DeviceArray<double> best_score;
    DeviceArray<unsigned long long> best_index;
    DeviceArray<unsigned char> record;
    PinnedArray<int64_t> h_stats;
    PinnedArray<unsigned char> h_record;
  } train;
  uint32_t train_n = 0;
  bool train_pending = false;
  struct UpdateBuffers {  // eg_update_device: scratch of the in-order update (update.cu) and its pinned host mirrors
    DeviceArray<EgUpdState> state;
    DeviceArray<EgUpdSlot> slots;
    DeviceArray<double> score, factors;
    DeviceArray<EgUpdPre> pre;
    DeviceArray<EgUpdCtl> ctl;
    DeviceArray<uint8_t> counts;
    PinnedArray<EgUpdState> h_state;
    PinnedArray<EgUpdSlot> h_slot;
    PinnedArray<EgUpdImprovement> h_imp;
  } upd;
  DeviceArray<EgUpdImprovement> upd_improvements;  // grown with the batch, at least EG_UPD_IMP_INLINE
  DeviceArray<double> suit_rows;       // scratch of the suitability kernel: crossing lists per site row
  DeviceArray<uint32_t> next_episode;  // work counter of the persistent episode kernels
};

namespace {

// ln(MAX_ACCEPTABLE_COST * 100 / MAX_ACCEPTABLE_COST) of the score, host libm (scoring.rs:13,32)
const double kLn100 = std::log(50000000000.0 * 100.0 / 50000000000.0);

// makes the context's device current: every entry point that touches device memory calls this before its first CUDA call
cudaError_t use_device(const eg_ctx* c) { return cudaSetDevice(c->device); }

template <typename T>
int upload(DeviceArray<T>& dst, const T* src, size_t n, cudaStream_t s) {
  // two spare elements, zeroed: the suitability kernel stages these arrays with bulk copies in 16-byte units
  EG_CUDA(dst.alloc(n + 2));
  EG_CUDA(cudaMemsetAsync(dst.get(), 0, (n + 2) * sizeof(T), s));
  if (n) EG_CUDA(cudaMemcpyAsync(dst.get(), src, n * sizeof(T), cudaMemcpyHostToDevice, s));
  return EG_OK;
}

int build_device_map(eg_ctx* c) {
  int rc = eg_host_map_validate(c->hmap);
  if (rc) return rc;
  EG_CUDA(use_device(c));
  c->map = eg_ctx::MapTables();  // the old tables go first
  c->map_ready = false;
  eg_host_build_tables(c->hmap, &c->htab);
  const EgHostMap& m = c->hmap;
  const int ns = m.grid_n * m.grid_n;
  const size_t n_lists = (size_t)EG_N_PCLASS * EG_NY * ns;
  cudaStream_t s = c->stream;
  eg_ctx::MapTables t;
  if ((rc = upload(t.small, &c->htab.small, 1, s))) return rc;
  if ((rc = upload(t.plant_terms, c->htab.plant_terms.data(), c->htab.plant_terms.size(), s))) return rc;
  if ((rc = upload(t.near, c->htab.near_factor.data(), c->htab.near_factor.size(), s))) return rc;
  if ((rc = upload(t.r2_limit, c->htab.r2_limit, (size_t)(2 * EG_N_RCLASS + 1), s))) return rc;
  if ((rc = upload(t.sx, m.sx.data(), m.sx.size(), s))) return rc;
  if ((rc = upload(t.sy, m.sy.data(), m.sy.size(), s))) return rc;
  if ((rc = upload(t.ex, m.ex.data(), m.ex.size(), s))) return rc;
  if ((rc = upload(t.ey, m.ey.data(), m.ey.size(), s))) return rc;
  if ((rc = upload(t.cx, m.cx.data(), m.cx.size(), s))) return rc;
  if ((rc = upload(t.cy, m.cy.data(), m.cy.size(), s))) return rc;
  if ((rc = upload(t.pop, c->htab.pop.data(), c->htab.pop.size(), s))) return rc;
  {
    std::vector<double> urban_r(c->htab.pop.size());
    for (size_t i = 0; i < urban_r.size(); i++) {
      urban_r[i] = std::sqrt((double)c->htab.pop[i]) * 5.0;
      t.urban_r_max = std::max(t.urban_r_max, urban_r[i]);
    }
    if ((rc = upload(t.urban_r, urban_r.data(), urban_r.size(), s))) return rc;
    EG_CUDA(cudaStreamSynchronize(s));  // urban_r is a local
  }
  DeviceArray<double> static_unsorted;  // [7][26][ns] static scores before the sort, needed by the build only
  EG_CUDA(t.site_opinion.alloc(ns));
  EG_CUDA(t.coast.alloc(ns));
  EG_CUDA(t.prefix.alloc((size_t)EG_N_RCLASS * EG_NY * ns));
  EG_CUDA(static_unsorted.alloc(n_lists));
  EG_CUDA(t.order.alloc(n_lists));
  EG_CUDA(t.walk.alloc(n_lists * 2));
  EgSiteBuildParams bp{};
  bp.grid_n = m.grid_n; bp.n_sites = ns; bp.step = m.step;
  bp.n_settlements = (int)m.sx.size(); bp.sx = t.sx.get(); bp.sy = t.sy.get(); bp.pop = t.pop.get();
  bp.n_existing = (int)m.ex.size(); bp.ex = t.ex.get(); bp.ey = t.ey.get();
  bp.n_coast = (int)m.cx.size(); bp.cx = t.cx.get(); bp.cy = t.cy.get();
  bp.size_factor = c->htab.small.size_factor;
  bp.prefix = t.prefix.get(); bp.coast_factor = t.coast.get(); bp.site_opinion = t.site_opinion.get();
  bp.static_unsorted = static_unsorted.get(); bp.order = t.order.get();
  bp.walk = (double2*)t.walk.get();
  int launches = 0;
  EG_CUDA(eg_build_site_tables(bp, s, &launches));
  c->launches += (uint64_t)launches;
  EG_CUDA(cudaStreamSynchronize(s));
  EgDeviceMap& d = c->dmap;
  d.small = t.small.get(); d.plant_terms = t.plant_terms.get(); d.near_geom = c->htab.near_geom;
  d.site_opinion = t.site_opinion.get(); d.coast_factor = t.coast.get(); d.order = t.order.get(); d.walk = t.walk.get();
  d.near_factor = t.near.get(); d.r2_limit = t.r2_limit.get(); d.r2_stride = c->htab.r2_stride;
  d.n_sites = ns; d.grid_n = m.grid_n; d.kmax = c->htab.kmax;
  c->map = std::move(t);
  c->map_ready = true;
  return EG_OK;
}

int ensure_scratch(eg_ctx* c, size_t n, bool sites, bool yearly, bool traj_in) {
  eg_ctx::Scratch& s = c->scratch;
  if (n > s.out.size()) EG_CUDA(s.out.alloc(n));
  if (n > s.traj.size()) EG_CUDA(s.traj.alloc(n));
  if (sites && n > s.sites.size()) EG_CUDA(s.sites.alloc(n));
  if (yearly && n > s.yearly.size()) EG_CUDA(s.yearly.alloc(n));
  if (traj_in && n > s.traj_in.size()) EG_CUDA(s.traj_in.alloc(n));
  return EG_OK;
}

// copies the first n episodes of the scratch outputs to the host buffers that are not NULL and waits for the copies
int copy_scratch_out(eg_ctx* c, uint32_t n, eg_result* out, eg_traj* traj_out, eg_sites* sites_out, eg_yearly* yearly_out) {
  const eg_ctx::Scratch& s = c->scratch;
  EG_CUDA(cudaMemcpyAsync(out, s.out.get(), (size_t)n * sizeof(eg_result), cudaMemcpyDeviceToHost, c->stream));
  if (traj_out) EG_CUDA(cudaMemcpyAsync(traj_out, s.traj.get(), (size_t)n * sizeof(eg_traj), cudaMemcpyDeviceToHost, c->stream));
  if (sites_out) EG_CUDA(cudaMemcpyAsync(sites_out, s.sites.get(), (size_t)n * sizeof(eg_sites), cudaMemcpyDeviceToHost, c->stream));
  if (yearly_out) EG_CUDA(cudaMemcpyAsync(yearly_out, s.yearly.get(), (size_t)n * sizeof(eg_yearly), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaStreamSynchronize(c->stream));
  return EG_OK;
}

int check_cfg(const eg_ctx* c, const eg_run_cfg* cfg) {
  if (!c) return eg_fail(EG_ERR_INVALID, "ctx is NULL");
  if (!cfg) return eg_fail(EG_ERR_INVALID, "cfg is NULL");
  if (!c->map_ready) return eg_fail(EG_ERR_STATE, "no map loaded: call eg_map_load or eg_map_set first");
  if (cfg->enable_construction_delays)
    return eg_fail(EG_ERR_INVALID,
                   "enable_construction_delays=1 is rejected: with delays on the reference's deficit handler cannot terminate "
                   "(a plant added in the loop is Planned, never active within the year, so remaining_deficit never shrinks; "
                   "simulation.rs:358-486, generator.rs:451-521) — see DESIGN.md section 9");
  return EG_OK;
}

EgEpisodeParams make_params(const eg_ctx* c, const eg_run_cfg* cfg, uint64_t seed, uint64_t first, uint32_t n) {
  EgEpisodeParams p{};
  p.map = c->dmap;
  p.policy = c->policy.d.get();
  p.seed = seed;
  p.first_episode = first;
  p.n = n;
  p.cost_only = cfg->cost_only;
  p.energy_sales = cfg->enable_energy_sales;
  p.same_stream = cfg->same_stream_all_episodes;
  p.replay_best = cfg->replay_best;
  p.count_weights = c->policy_count_weights ? 1u : 0u;
  p.stagnation = c->policy_stagnation ? 1u : 0u;
  p.ln100 = kLn100;
  p.next_episode = c->next_episode.get();
  p.nf_entries = c->htab.r2_limit[2 * EG_N_RCLASS];
  return p;
}

EgSuitabilityParams suitability_params(const eg_ctx* c, int use_loaded_map, int mode, int half, int side, double step, uint32_t year_first,
                                       uint32_t n_years, uint32_t first, uint32_t n, double* d_scores) {
  EgSuitabilityParams p{};
  p.mode = mode; p.half = half; p.side = side; p.step = step; p.first = first; p.n = n;
  p.year_first = (int)year_first; p.n_years = (int)n_years;
  p.n_settlements = use_loaded_map ? (int)c->hmap.sx.size() : 0;
  p.sx = c->map.sx.get(); p.sy = c->map.sy.get(); p.pop = c->map.pop.get(); p.urban_r = c->map.urban_r.get(); p.urban_r_max = c->map.urban_r_max;
  p.n_generators = use_loaded_map ? (int)c->hmap.ex.size() : 0;
  p.gx = c->map.ex.get(); p.gy = c->map.ey.get();
  p.n_coast = (int)c->hmap.cx.size(); p.cx = c->map.cx.get(); p.cy = c->map.cy.get();
  p.scores = d_scores;
  return p;
}

// grows the kernel's scratch to what the launch needs, then queues the launch
int launch_suitability(eg_ctx* c, const EgSuitabilityParams& p) {
  const size_t rows = eg_suitability_rows_bytes(p.mode == 0 ? 2 * p.half + 1 : p.side) / sizeof(double);
  if (rows > c->suit_rows.size()) EG_CUDA(c->suit_rows.alloc(rows));
  EG_CUDA(eg_launch_suitability(p, c->suit_rows.get(), c->stream));
  if (p.n && p.n_years) c->launches += 2;
  return EG_OK;
}

// runs the kernel into a temporary device buffer and copies the scores to the host
int suitability_to_host(eg_ctx* c, EgSuitabilityParams p, double* scores_out) {
  EG_CUDA(use_device(c));
  const size_t count = (size_t)p.n * p.n_years * EG_NT;
  DeviceArray<double> d_scores;
  EG_CUDA(d_scores.alloc(std::max<size_t>(count, 1)));
  p.scores = d_scores.get();
  const int rc = launch_suitability(c, p);
  if (rc) return rc;
  EG_CUDA(cudaMemcpyAsync(scores_out, d_scores.get(), count * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaStreamSynchronize(c->stream));
  return EG_OK;
}

// argument checks of eg_location_analysis_sites and eg_location_analysis_sites_device (`name`)
int check_sites_args(const eg_ctx* c, const double* scores, const char* name, uint32_t sites_per_axis, uint32_t year_first,
                     uint32_t n_years, uint32_t first_site, uint32_t n_sites) {
  if (!c || !scores) return eg_fail(EG_ERR_INVALID, std::string(name) + ": NULL argument");
  if (!c->map_ready) return eg_fail(EG_ERR_STATE, "no map loaded (the coastline polygon is needed)");
  if (year_first >= EG_NY || n_years > EG_NY - year_first) return eg_fail(EG_ERR_INVALID, "year range outside 2025..2050");
  if (sites_per_axis == 0 || sites_per_axis > 65535u) return eg_fail(EG_ERR_INVALID, "sites_per_axis out of range");
  if ((uint64_t)first_site + n_sites > (uint64_t)sites_per_axis * sites_per_axis) return eg_fail(EG_ERR_INVALID, "site range exceeds the grid");
  return EG_OK;
}

}  // namespace

extern "C" {

const char* eg_last_error(void) { return g_last_error.c_str(); }

int eg_init(int device, void* cuda_stream, eg_ctx** out) {
  if (!out) return eg_fail(EG_ERR_INVALID, "eg_init: out is NULL");
  int count = 0;
  cudaError_t err = cudaGetDeviceCount(&count);
  if (err != cudaSuccess || count == 0)
    return eg_fail(EG_ERR_NO_DEVICE, std::string("no CUDA device (") + cudaGetErrorString(err) + "); eirgrid_b200 has no CPU fallback");
  if (device < 0 || device >= count) return eg_fail(EG_ERR_INVALID, "eg_init: device index out of range");
  EG_CUDA(cudaSetDevice(device));
  std::unique_ptr<eg_ctx> c(new eg_ctx());
  c->device = device;
  c->stream = (cudaStream_t)cuda_stream;
  if (!cuda_stream) {
    err = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (err != cudaSuccess) return eg_fail(EG_ERR_CUDA, cudaGetErrorString(err));
    c->own_stream.reset(c->stream);
  }
  err = c->next_episode.alloc(1);
  if (err != cudaSuccess) return eg_fail(EG_ERR_CUDA, cudaGetErrorString(err));
  *out = c.release();
  return EG_OK;
}

void eg_destroy(eg_ctx* c) {
  if (!c) return;
  use_device(c);
  cudaStreamSynchronize(c->stream);
  delete c;
}

int eg_sync(eg_ctx* c) {
  if (!c) return eg_fail(EG_ERR_INVALID, "ctx is NULL");
  EG_CUDA(cudaStreamSynchronize(c->stream));
  return EG_OK;
}

uint64_t eg_kernel_launches(const eg_ctx* c) { return c ? c->launches : 0; }

int eg_map_load(eg_ctx* c, const char* settlements_json, const char* generators_csv, const char* coastline_json) {
  if (!c || !settlements_json || !generators_csv || !coastline_json) return eg_fail(EG_ERR_INVALID, "eg_map_load: NULL argument");
  int rc = eg_host_map_load(&c->hmap, settlements_json, generators_csv, coastline_json);
  if (rc) return rc;
  return build_device_map(c);
}

int eg_map_set(eg_ctx* c, const eg_map_desc* desc) {
  if (!c) return eg_fail(EG_ERR_INVALID, "eg_map_set: ctx is NULL");
  int rc = eg_host_map_set(&c->hmap, desc);
  if (rc) return rc;
  return build_device_map(c);
}

int eg_map_info(const eg_ctx* c, uint32_t out[4]) {
  if (!c || !out) return eg_fail(EG_ERR_INVALID, "eg_map_info: NULL argument");
  if (!c->map_ready) return eg_fail(EG_ERR_STATE, "no map loaded");
  out[0] = (uint32_t)c->hmap.sx.size();
  out[1] = (uint32_t)c->hmap.ex.size();
  out[2] = (uint32_t)c->hmap.cx.size();
  out[3] = (uint32_t)c->hmap.grid_n;
  return EG_OK;
}

int eg_map_site_tables(eg_ctx* c, uint32_t year_index, uint32_t rclass, uint32_t pclass, double* prefix_score,
                       double* static_score_sorted, uint32_t* order_sorted) {
  if (!c) return eg_fail(EG_ERR_INVALID, "ctx is NULL");
  if (!c->map_ready) return eg_fail(EG_ERR_STATE, "no map loaded");
  if (year_index >= EG_NY || rclass >= EG_N_RCLASS || pclass >= EG_N_PCLASS) return eg_fail(EG_ERR_INVALID, "index out of range");
  const size_t ns = (size_t)c->dmap.n_sites;
  const size_t list = ((size_t)pclass * EG_NY + year_index) * ns;
  EG_CUDA(use_device(c));
  if (prefix_score)
    EG_CUDA(cudaMemcpyAsync(prefix_score, c->map.prefix.get() + ((size_t)rclass * EG_NY + year_index) * ns, ns * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  if (static_score_sorted)  // the static score is the first half of each walk entry
    EG_CUDA(cudaMemcpy2DAsync(static_score_sorted, sizeof(double), c->map.walk.get() + 2 * list, 2 * sizeof(double), sizeof(double), ns,
                              cudaMemcpyDeviceToHost, c->stream));
  std::vector<uint16_t> tmp;
  if (order_sorted) {
    tmp.resize(ns);
    EG_CUDA(cudaMemcpyAsync(tmp.data(), c->map.order.get() + list, ns * sizeof(uint16_t), cudaMemcpyDeviceToHost, c->stream));
  }
  EG_CUDA(cudaStreamSynchronize(c->stream));
  if (order_sorted)
    for (size_t i = 0; i < ns; i++) order_sorted[i] = (uint32_t)(tmp[i] >> 8) * (uint32_t)c->dmap.grid_n + (tmp[i] & 0xFFu);
  return EG_OK;
}

int eg_map_site_static(eg_ctx* c, double* coast_factor, double* site_opinion) {
  if (!c) return eg_fail(EG_ERR_INVALID, "ctx is NULL");
  if (!c->map_ready) return eg_fail(EG_ERR_STATE, "no map loaded");
  const size_t ns = (size_t)c->dmap.n_sites;
  EG_CUDA(use_device(c));
  if (coast_factor) EG_CUDA(cudaMemcpyAsync(coast_factor, c->map.coast.get(), ns * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  if (site_opinion) EG_CUDA(cudaMemcpyAsync(site_opinion, c->map.site_opinion.get(), ns * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaStreamSynchronize(c->stream));
  return EG_OK;
}

int eg_weights_upload(eg_ctx* c, const eg_weights* w) {
  if (!c || !w) return eg_fail(EG_ERR_INVALID, "eg_weights_upload: NULL argument");
  EG_CUDA(use_device(c));
  if (!c->policy.d.get()) {
    eg_ctx::PolicyBuffers p;
    EG_CUDA(p.d.alloc(1));
    for (int b = 0; b < 2; b++) {
      EG_CUDA(p.h[b].alloc(1));
      cudaEvent_t e = nullptr;
      EG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      p.copied[b].reset(e);
    }
    c->policy = std::move(p);
  }
  // two pinned staging buffers used in turn: the copy is queued on the stream and the call returns without waiting for it;
  // a buffer is refilled only after the copy issued from it two uploads ago has completed (normally long ago)
  const int b = c->policy_turn;
  c->policy_turn ^= 1;
  EG_CUDA(cudaEventSynchronize(c->policy.copied[b].get()));
  EgPolicyDevice& pol = *c->policy.h[b].get();
  if (!eg_weights_fill_policy(*w, &pol))
    return eg_fail(EG_ERR_OVERFLOW, "eg_weights_upload: the best-strategy lists exceed the device snapshot's capacity (EG_BEST_CAPACITY / EG_TRAJ_CAPACITY actions)");
  EG_CUDA(cudaMemcpyAsync(c->policy.d.get(), &pol, sizeof(pol), cudaMemcpyHostToDevice, c->stream));
  EG_CUDA(cudaEventRecord(c->policy.copied[b].get(), c->stream));
  c->policy_ready = true;
  c->policy_count_weights = pol.has_count_weights != 0;
  c->policy_stagnation = pol.iwi > 500;
  return EG_OK;
}

int eg_rollout_batch_device(eg_ctx* c, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode, uint32_t n,
                            eg_result* d_out, eg_traj* d_traj, eg_sites* d_sites, eg_yearly* d_yearly) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!c->policy_ready) return eg_fail(EG_ERR_STATE, "no weights uploaded: call eg_weights_upload first");
  if (!d_out) return eg_fail(EG_ERR_INVALID, "eg_rollout_batch_device: d_out is NULL");
  EG_CUDA(use_device(c));
  EgEpisodeParams p = make_params(c, cfg, seed, first_episode, n);
  p.out = d_out; p.traj = d_traj; p.sites = d_sites; p.yearly = d_yearly;
  EG_CUDA(eg_launch_rollout(p, c->stream));
  if (n) c->launches++;
  return EG_OK;
}

int eg_rollout_batch(eg_ctx* c, const eg_weights* w, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode,
                     uint32_t n, eg_result* out, eg_traj* traj_out, eg_sites* sites_out, eg_yearly* yearly_out) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!w || !out) return eg_fail(EG_ERR_INVALID, "eg_rollout_batch: NULL argument");
  EG_CUDA(use_device(c));
  if ((rc = eg_weights_upload(c, w))) return rc;
  if ((rc = ensure_scratch(c, n, sites_out != nullptr, yearly_out != nullptr, false))) return rc;
  const eg_ctx::Scratch& s = c->scratch;
  rc = eg_rollout_batch_device(c, cfg, seed, first_episode, n, s.out.get(), traj_out ? s.traj.get() : nullptr,
                               sites_out ? s.sites.get() : nullptr, yearly_out ? s.yearly.get() : nullptr);
  if (rc) return rc;
  return copy_scratch_out(c, n, out, traj_out, sites_out, yearly_out);
}

int eg_replay_batch_device(eg_ctx* c, const eg_run_cfg* cfg, const eg_traj* d_in, uint32_t n, eg_result* d_out,
                           eg_sites* d_sites, eg_yearly* d_yearly) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!d_in || !d_out) return eg_fail(EG_ERR_INVALID, "eg_replay_batch_device: NULL argument");
  EG_CUDA(use_device(c));
  EgEpisodeParams p = make_params(c, cfg, 0, 0, n);
  p.policy = nullptr;
  p.replay_in = d_in;
  p.out = d_out; p.traj = nullptr; p.sites = d_sites; p.yearly = d_yearly;
  EG_CUDA(eg_launch_replay(p, c->stream));
  if (n) c->launches++;
  return EG_OK;
}

int eg_replay_batch(eg_ctx* c, const eg_run_cfg* cfg, const eg_traj* in, uint32_t n, eg_result* out, eg_sites* sites_out,
                    eg_yearly* yearly_out) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!in || !out) return eg_fail(EG_ERR_INVALID, "eg_replay_batch: NULL argument");
  EG_CUDA(use_device(c));
  if ((rc = ensure_scratch(c, n, sites_out != nullptr, yearly_out != nullptr, true))) return rc;
  const eg_ctx::Scratch& s = c->scratch;
  EG_CUDA(cudaMemcpyAsync(s.traj_in.get(), in, (size_t)n * sizeof(eg_traj), cudaMemcpyHostToDevice, c->stream));
  rc = eg_replay_batch_device(c, cfg, s.traj_in.get(), n, s.out.get(), sites_out ? s.sites.get() : nullptr, yearly_out ? s.yearly.get() : nullptr);
  if (rc) return rc;
  return copy_scratch_out(c, n, out, nullptr, sites_out, yearly_out);
}

int eg_update_stats_device(eg_ctx* c, const eg_weights* w, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n,
                           int64_t* d_stats, double* d_best_score, unsigned long long* d_best_index) {
  if (!c || !w || !d_results || !d_trajs || !d_stats || !d_best_score || !d_best_index)
    return eg_fail(EG_ERR_INVALID, "eg_update_stats_device: NULL argument");
  if (!c->policy_ready) return eg_fail(EG_ERR_STATE, "no weights uploaded: call eg_weights_upload first");
  EG_CUDA(use_device(c));
  EgStatsParams p{};
  p.consts = eg_contrast_consts(*w);
  p.policy = c->policy.d.get();
  p.results = d_results; p.trajs = d_trajs; p.n = n;
  p.stats = d_stats; p.best_score = d_best_score; p.best_index = d_best_index;
  p.ln100 = kLn100;
  EG_CUDA(eg_launch_stats(p, c->stream));
  c->launches += n ? 3 : 1;  // reset + accumulate + arg-best kernels
  return EG_OK;
}

int eg_update_stats_clear_device(eg_ctx* c, int64_t* d_stats) {
  if (!c || !d_stats) return eg_fail(EG_ERR_INVALID, "eg_update_stats_clear_device: NULL argument");
  EG_CUDA(use_device(c));
  EG_CUDA(cudaMemsetAsync(d_stats, 0, (size_t)EG_STATS_WORDS * sizeof(int64_t), c->stream));
  return EG_OK;
}

int eg_update_pack_best_device(eg_ctx* c, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n, const double* d_best_score,
                               const unsigned long long* d_best_index, uint64_t first_global_episode, void* d_record) {
  if (!c || !d_results || !d_trajs || !d_best_score || !d_best_index || !d_record)
    return eg_fail(EG_ERR_INVALID, "eg_update_pack_best_device: NULL argument");
  EG_CUDA(use_device(c));
  EG_CUDA(eg_launch_pack_best(d_results, d_trajs, n, d_best_score, d_best_index, first_global_episode, d_record, c->stream));
  c->launches++;
  return EG_OK;
}

int eg_update_pack_exchange_device(eg_ctx* c, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n, const int64_t* d_stats,
                                   const double* d_best_score, const unsigned long long* d_best_index, uint64_t first_global_episode,
                                   const uint64_t* peer_buffers, const uint64_t* peer_flags, uint32_t world, uint32_t rank, uint32_t epoch,
                                   uint32_t* d_error) {
  if (!c || !d_results || !d_trajs || !d_stats || !d_best_score || !d_best_index || !peer_buffers || !peer_flags || !d_error)
    return eg_fail(EG_ERR_INVALID, "eg_update_pack_exchange_device: NULL argument");
  if (world == 0 || world > EG_MAX_PEERS || rank >= world) return eg_fail(EG_ERR_INVALID, "eg_update_pack_exchange_device: bad world / rank");
  EG_CUDA(use_device(c));
  EgExchangeParams p{};
  p.results = d_results; p.trajs = d_trajs; p.n = n; p.best_score = d_best_score; p.best_index = d_best_index;
  p.first_global = first_global_episode; p.stats = d_stats; p.world = world; p.rank = rank; p.epoch = epoch; p.error = d_error;
  for (uint32_t r = 0; r < world; r++) { p.peer_buf[r] = peer_buffers[r]; p.peer_flag[r] = peer_flags[r]; }
  EG_CUDA(eg_launch_pack_exchange(p, c->stream));
  c->launches++;
  return EG_OK;
}

int eg_train_batch_begin(eg_ctx* c, const eg_weights* w, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode, uint32_t n) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!w) return eg_fail(EG_ERR_INVALID, "eg_train_batch_begin: weights are NULL");
  if (c->train_pending) return eg_fail(EG_ERR_STATE, "eg_train_batch_begin: a batch is already in flight on this context");
  EG_CUDA(use_device(c));
  if (!c->train.stats.get()) {
    eg_ctx::TrainBuffers t;
    EG_CUDA(t.stats.alloc(EG_STATS_WORDS));
    EG_CUDA(t.best_score.alloc(1));
    EG_CUDA(t.best_index.alloc(1));
    EG_CUDA(t.record.alloc(EG_BEST_RECORD_BYTES));
    EG_CUDA(t.h_stats.alloc(EG_STATS_WORDS));
    EG_CUDA(t.h_record.alloc(EG_BEST_RECORD_BYTES));
    c->train = std::move(t);
  }
  if ((rc = eg_weights_upload(c, w))) return rc;
  if ((rc = ensure_scratch(c, n, false, false, false))) return rc;
  const eg_ctx::Scratch& s = c->scratch;
  const eg_ctx::TrainBuffers& t = c->train;
  if ((rc = eg_rollout_batch_device(c, cfg, seed, first_episode, n, s.out.get(), s.traj.get(), nullptr, nullptr))) return rc;
  if ((rc = eg_update_stats_clear_device(c, t.stats.get()))) return rc;
  if ((rc = eg_update_stats_device(c, w, s.out.get(), s.traj.get(), n, t.stats.get(), t.best_score.get(), t.best_index.get()))) return rc;
  if ((rc = eg_update_pack_best_device(c, s.out.get(), s.traj.get(), n, t.best_score.get(), t.best_index.get(), first_episode, t.record.get()))) return rc;
  EG_CUDA(cudaMemcpyAsync(t.h_stats.get(), t.stats.get(), EG_STATS_WORDS * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaMemcpyAsync(t.h_record.get(), t.record.get(), EG_BEST_RECORD_BYTES, cudaMemcpyDeviceToHost, c->stream));
  c->train_n = n;
  c->train_pending = true;
  return EG_OK;
}

int eg_train_batch_end(eg_ctx* c, int64_t* stats_out, void* record_out) {
  if (!c || !stats_out || !record_out) return eg_fail(EG_ERR_INVALID, "eg_train_batch_end: NULL argument");
  if (!c->train_pending) return eg_fail(EG_ERR_STATE, "eg_train_batch_end: no batch in flight");
  EG_CUDA(use_device(c));
  c->train_pending = false;
  EG_CUDA(cudaStreamSynchronize(c->stream));
  std::memcpy(stats_out, c->train.h_stats.get(), EG_STATS_WORDS * sizeof(int64_t));
  std::memcpy(record_out, c->train.h_record.get(), EG_BEST_RECORD_BYTES);
  return EG_OK;
}

int eg_train_batch_results(eg_ctx* c, eg_result* out, eg_traj* traj_out) {
  if (!c || !out) return eg_fail(EG_ERR_INVALID, "eg_train_batch_results: NULL argument");
  if (c->train_pending || !c->train_n) return eg_fail(EG_ERR_STATE, "eg_train_batch_results: no finished batch");
  EG_CUDA(use_device(c));
  return copy_scratch_out(c, c->train_n, out, traj_out, nullptr, nullptr);
}

// ---- in-order update on the device (update.cu) ----------------------------------------------------------------------
int eg_update_device(eg_ctx* c, eg_weights* w, const eg_result* d_results, const eg_traj* d_trajs, uint32_t n, uint32_t replay_best,
                     uint64_t rng_seed, eg_update_stats* stats_out) {
  if (!c || !w || (n && (!d_results || !d_trajs))) return eg_fail(EG_ERR_INVALID, "eg_update_device: NULL argument");
  EG_CUDA(use_device(c));
  if (!c->upd.state.get()) {
    eg_ctx::UpdateBuffers u;
    EG_CUDA(u.state.alloc(1));
    EG_CUDA(u.slots.alloc((size_t)EG_UPD_CHUNK + 1));
    EG_CUDA(u.score.alloc(EG_UPD_CHUNK));
    EG_CUDA(u.pre.alloc(EG_UPD_CHUNK));
    EG_CUDA(u.ctl.alloc(EG_UPD_CHUNK));
    EG_CUDA(u.counts.alloc((size_t)EG_NY * EG_UPD_CHUNK * EG_UPD_ROW));
    EG_CUDA(u.factors.alloc((size_t)EG_NY * EG_UPD_CHUNK * EG_UPD_ENTRIES));
    EG_CUDA(u.h_state.alloc(1));
    EG_CUDA(u.h_slot.alloc(1));
    EG_CUDA(u.h_imp.alloc(EG_UPD_IMP_INLINE));
    c->upd = std::move(u);
  }
  if (n > c->upd_improvements.size()) EG_CUDA(c->upd_improvements.alloc(std::max<uint32_t>(n, EG_UPD_IMP_INLINE)));
  const eg_ctx::UpdateBuffers& u = c->upd;
  const EgUpdBuffers view{u.state.get(), u.slots.get(), u.score.get(), u.pre.get(), u.ctl.get(), u.counts.get(), u.factors.get(),
                          c->upd_improvements.get(), (uint32_t)c->upd_improvements.size()};
  // the pinned mirrors are free again: every call ends with a stream synchronisation
  if (!eg_weights_fill_update_state(*w, u.h_state.get(), u.h_slot.get()))
    return eg_fail(EG_ERR_OVERFLOW, "eg_update_device: the best-strategy lists exceed EG_UPD_CAT_CAPACITY entries");
  const uint32_t iteration0 = w->iteration_count;
  EG_CUDA(cudaMemcpyAsync(view.state, u.h_state.get(), sizeof(EgUpdState), cudaMemcpyHostToDevice, c->stream));
  EG_CUDA(cudaMemcpyAsync(view.slots, u.h_slot.get(), sizeof(EgUpdSlot), cudaMemcpyHostToDevice, c->stream));
  for (uint32_t base = 0; base < n; base += EG_UPD_CHUNK) {
    const uint32_t cnt = std::min<uint32_t>(EG_UPD_CHUNK, n - base);
    int launches = 0;
    EG_CUDA(eg_launch_update_pass(view, d_results + base, d_trajs + base, cnt, base, replay_best, rng_seed, c->stream, &launches));
    c->launches += (uint64_t)launches;
  }
  EG_CUDA(cudaMemcpyAsync(u.h_state.get(), view.state, sizeof(EgUpdState), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaMemcpyAsync(u.h_slot.get(), view.slots, sizeof(EgUpdSlot), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaMemcpyAsync(u.h_imp.get(), view.improvements, (size_t)EG_UPD_IMP_INLINE * sizeof(EgUpdImprovement), cudaMemcpyDeviceToHost, c->stream));
  EG_CUDA(cudaStreamSynchronize(c->stream));
  const EgUpdState& st = *u.h_state.get();
  std::vector<EgUpdImprovement> more;
  const EgUpdImprovement* imps = u.h_imp.get();
  if (st.n_improvements > EG_UPD_IMP_INLINE) {  // rare: more improving episodes than the inline window
    more.resize(st.n_improvements);
    EG_CUDA(cudaMemcpyAsync(more.data(), view.improvements, (size_t)st.n_improvements * sizeof(EgUpdImprovement), cudaMemcpyDeviceToHost, c->stream));
    EG_CUDA(cudaStreamSynchronize(c->stream));
    imps = more.data();
  }
  eg_weights_apply_update_state(*w, st, *u.h_slot.get(), imps, st.n_improvements, iteration0);
  if (stats_out) {
    eg_update_stats so;
    std::memset(&so, 0, sizeof(so));
    so.n_episodes = n;
    so.n_improvements = st.n_improvements;
    so.n_contrast_applied = st.n_applied;
    so.iterations_without_improvement = st.iwi;
    so.best_score = st.has_best ? st.best_score : 0.0;
    so.batch_best_score = st.batch_best_index >= 0 ? st.batch_best_score : 0.0;
    so.batch_best_episode = st.batch_best_index;
    so.n_flagged = st.n_flagged;
    *stats_out = so;
  }
  return EG_OK;
}

int eg_train_batch_inorder(eg_ctx* c, eg_weights* w, const eg_run_cfg* cfg, uint64_t seed, uint64_t first_episode, uint32_t n,
                           uint64_t rng_seed, eg_update_stats* stats_out) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!w) return eg_fail(EG_ERR_INVALID, "eg_train_batch_inorder: weights are NULL");
  if (c->train_pending) return eg_fail(EG_ERR_STATE, "eg_train_batch_inorder: a batch is already in flight on this context");
  EG_CUDA(use_device(c));
  if ((rc = eg_weights_upload(c, w))) return rc;
  if ((rc = ensure_scratch(c, n, false, false, false))) return rc;
  const eg_ctx::Scratch& s = c->scratch;
  if ((rc = eg_rollout_batch_device(c, cfg, seed, first_episode, n, s.out.get(), s.traj.get(), nullptr, nullptr))) return rc;
  c->train_n = n;
  return eg_update_device(c, w, s.out.get(), s.traj.get(), n, cfg->replay_best, rng_seed, stats_out);
}

// ---- CSV export of the best run (utils/csv_export.rs): the replay here, the files in report_files.cpp ----------------
int eg_export_best_run_csv(eg_ctx* c, const eg_weights* w, const eg_run_cfg* cfg, const char* output_dir, char* written_dir) {
  int rc = check_cfg(c, cfg);
  if (rc) return rc;
  if (!w || !output_dir) return eg_fail(EG_ERR_INVALID, "eg_export_best_run_csv: NULL argument");
  if (!w->has_best) return eg_fail(EG_ERR_STATE, "eg_export_best_run_csv: the weights hold no best strategy yet");
  // the best run as a record: best_actions[y] = deficit actions followed by the additional actions (Appendix C of SURVEY.md)
  eg_traj traj;
  std::memset(&traj, 0, sizeof(traj));
  int row[EG_NY + 1];  // first slot of each year's row in the record
  row[0] = 0;
  for (int y = 0; y < EG_NY; y++) {
    const size_t n = std::min<size_t>(w->best_actions[y].size(), (size_t)(EG_TRAJ_CAPACITY - row[y]));
    const size_t nd = std::min<size_t>(w->best_deficit_actions[y].size(), n);
    traj.n_deficit[y] = (uint16_t)nd;
    traj.n_additional[y] = (uint16_t)(n - nd);
    for (size_t i = 0; i < n; i++) traj.actions[row[y] + i] = w->best_actions[y][i];
    row[y + 1] = row[y] + (int)n;
  }
  eg_result res;
  eg_yearly yearly;
  eg_run_cfg rcfg = *cfg;
  rcfg.replay_best = 0;
  eg_sites sites;
  if ((rc = eg_replay_batch(c, &rcfg, &traj, 1, &res, &sites, &yearly))) return rc;
  return eg_write_best_run_csv(output_dir, w, c->hmap, c->htab, traj, row, res, yearly, sites, written_dir);
}

int eg_location_analysis(eg_ctx* c, int use_loaded_map, int32_t half_steps, double step, double* scores_out,
                         uint32_t first_point, uint32_t n_points) {
  return eg_location_analysis_year(c, use_loaded_map, 0, half_steps, step, scores_out, first_point, n_points);
}

int eg_location_analysis_year(eg_ctx* c, int use_loaded_map, uint32_t year_index, int32_t half_steps, double step, double* scores_out,
                              uint32_t first_point, uint32_t n_points) {
  if (!c || !scores_out) return eg_fail(EG_ERR_INVALID, "eg_location_analysis: NULL argument");
  if (year_index >= EG_NY) return eg_fail(EG_ERR_INVALID, "eg_location_analysis_year: year_index out of range");
  if (!c->map_ready) return eg_fail(EG_ERR_STATE, "no map loaded (the coastline polygon is needed)");
  if (half_steps < 0 || half_steps > 1000) return eg_fail(EG_ERR_INVALID, "half_steps out of range");
  const uint32_t side = (uint32_t)(2 * half_steps + 1);
  if ((uint64_t)first_point + n_points > (uint64_t)side * side) return eg_fail(EG_ERR_INVALID, "point range exceeds the analysis grid");
  return suitability_to_host(c, suitability_params(c, use_loaded_map, 0, half_steps, 0, step, year_index, 1, first_point, n_points, nullptr), scores_out);
}

int eg_location_analysis_sites_device(eg_ctx* c, int use_loaded_map, uint32_t sites_per_axis, double step, uint32_t year_first,
                                      uint32_t n_years, uint32_t first_site, uint32_t n_sites, double* d_scores) {
  const int rc = check_sites_args(c, d_scores, "eg_location_analysis_sites_device", sites_per_axis, year_first, n_years, first_site, n_sites);
  if (rc) return rc;
  EG_CUDA(use_device(c));
  return launch_suitability(c, suitability_params(c, use_loaded_map, 1, 0, (int)sites_per_axis, step, year_first, n_years, first_site, n_sites, d_scores));
}

int eg_location_analysis_sites(eg_ctx* c, int use_loaded_map, uint32_t sites_per_axis, double step, uint32_t year_first, uint32_t n_years,
                               uint32_t first_site, uint32_t n_sites, double* scores_out) {
  const int rc = check_sites_args(c, scores_out, "eg_location_analysis_sites", sites_per_axis, year_first, n_years, first_site, n_sites);
  if (rc) return rc;
  return suitability_to_host(c, suitability_params(c, use_loaded_map, 1, 0, (int)sites_per_axis, step, year_first, n_years, first_site, n_sites, nullptr), scores_out);
}

// LocationAnalysis::analyze_map + save_cache + save_to_file (map_handler.rs:61-142,208-248; bin/analyze_locations.rs:19-46)
int eg_location_analysis_write(eg_ctx* c, int use_loaded_map, double min_suitability, const char* cache_dir, const char* text_path) {
  if (!c) return eg_fail(EG_ERR_INVALID, "eg_location_analysis_write: ctx is NULL");
  const int half = 25;          // ceil(MAP_MAX_X / (2 * GRID_CELL_SIZE)) = ceil(50000 / 2000)
  const double step = 2000.0;   // GRID_CELL_SIZE * 2
  const int side = 2 * half + 1;
  std::vector<double> scores((size_t)side * side * EG_NT);
  int rc = eg_location_analysis_year(c, use_loaded_map, 0, half, step, scores.data(), 0, (uint32_t)(side * side));
  if (rc) return rc;
  return eg_write_location_analysis(scores, half, step, min_suitability, cache_dir, text_path);
}

}  // extern "C"
