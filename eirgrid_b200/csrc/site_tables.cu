// site_tables.cu — static candidate-site tables, built on the GPU once per map (sm_100a).
//
// Replaces the per-call work of MetalLocationSearch::find_suitable_location's CPU branch
// (gpu/metal_location_search.rs:110-176, called from Map::find_best_generator_location,
// utils/map_handler.rs:1133-1143) that does not depend on the episode:
//   * the settlement product  prod_s (1 + pop_s/1e6) / (1 + d_s/1e4)     (:130-134), per year because pop_s grows
//   * the penalty of the plants that exist before the simulation starts  (:137-150), they head Map.generators
//   * the coastline factor 1/(1 + min_d/5000)                            (:153-163)
//   * the size factor                                                     (:166)
// and the per-site settlement opinion of Map::calc_new_generator_opinion (map_handler.rs:931-941).
// One thread per (site, year) multiplies in the reference's order (settlements, then plants, in list order), so the
// products round exactly as the reference's. Sites are then ranked per (placement class, year) by static score.
// Compiled with --fmad=false.
#include "site_tables.cuh"
#include "tables.h"

namespace {

__constant__ double c_radii[EG_N_RCLASS] = {3000.0, 5000.0, 6000.0, 7000.0, 8000.0, 12000.0};
__constant__ int c_pc_rclass[EG_N_PCLASS] = {0, 1, 1, 2, 3, 4, 5};
__constant__ int c_pc_water[EG_N_PCLASS] = {0, 0, 1, 1, 0, 0, 0};

__device__ __forceinline__ double clamp_map(double v) { return fmin(fmax(v, 0.0), 50000.0); }  // Coordinate::new, data/poi.rs:11-15

// grid: (ceil(n_sites/128), 26)
__global__ void __launch_bounds__(128) eg_site_prefix_kernel(const EgSiteBuildParams p) {
  const int site = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (site >= p.n_sites) return;
  const int i = site / p.grid_n, j = site - i * p.grid_n;
  const double lx = clamp_map((double)i * p.step), ly = clamp_map((double)j * p.step);
  const uint32_t* __restrict__ pop = p.pop + (size_t)y * p.n_settlements;
  double score = 1.0;
  for (int s = 0; s < p.n_settlements; s++) {
    const double dx = lx - __ldg(&p.sx[s]), dy = ly - __ldg(&p.sy[s]);
    const double distance = sqrt(dx * dx + dy * dy);
    const double population_factor = (double)__ldg(&pop[s]) / 1000000.0;
    score *= (1.0 + population_factor) / (1.0 + distance / 10000.0);
  }
  double sc[EG_N_RCLASS];
#pragma unroll
  for (int rc = 0; rc < EG_N_RCLASS; rc++) sc[rc] = score;
  for (int g = 0; g < p.n_existing; g++) {
    const double dx = lx - __ldg(&p.ex[g]), dy = ly - __ldg(&p.ey[g]);
    const double distance = sqrt(dx * dx + dy * dy);
#pragma unroll
    for (int rc = 0; rc < EG_N_RCLASS; rc++)
      if (distance < c_radii[rc]) sc[rc] *= distance / c_radii[rc];
  }
#pragma unroll
  for (int rc = 0; rc < EG_N_RCLASS; rc++) p.prefix[((size_t)rc * EG_NY + y) * p.n_sites + site] = sc[rc];

  if (y == 0) {
    double mind = 1.7976931348623157e308;
    for (int c = 0; c < p.n_coast; c++) {
      const double dx = lx - __ldg(&p.cx[c]), dy = ly - __ldg(&p.cy[c]);
      const double d = sqrt(dx * dx + dy * dy);
      if (c == 0 || d < mind) mind = d;
    }
    p.coast_factor[site] = 1.0 / (1.0 + mind / 5000.0);
    double sum = 0.0;
    for (int s = 0; s < p.n_settlements; s++) {
      const double dx = __ldg(&p.sx[s]) - lx, dy = __ldg(&p.sy[s]) - ly;
      sum += 1.0 / (1.0 + sqrt(dx * dx + dy * dy) / 10000.0);  // Settlement::calc_range_opinion, settlement.rs:103-106
    }
    p.site_opinion[site] = p.n_settlements ? sum / (double)p.n_settlements : 1.0;
  }
}

// grid: (ceil(n_sites/128), 26, 7)
__global__ void __launch_bounds__(128) eg_site_static_kernel(const EgSiteBuildParams p) {
  const int site = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y, pc = blockIdx.z;
  if (site >= p.n_sites) return;
  double score = p.prefix[((size_t)c_pc_rclass[pc] * EG_NY + y) * p.n_sites + site];
  if (c_pc_water[pc]) score *= p.coast_factor[site];
  score *= p.size_factor;
  p.static_unsorted[((size_t)pc * EG_NY + y) * p.n_sites + site] = score;
}

// Rank sort per (pclass, year) list: rank = number of sites that precede this one in (score desc, site asc) order.
// grid: (ceil(n_sites/256), 26, 7); the list is streamed through shared memory in tiles of 256.
__global__ void __launch_bounds__(256) eg_site_rank_kernel(const EgSiteBuildParams p) {
  __shared__ double tile[256];
  const int y = blockIdx.y, pc = blockIdx.z;
  const size_t base = ((size_t)pc * EG_NY + y) * p.n_sites;
  const double* __restrict__ s = p.static_unsorted + base;
  const int me = blockIdx.x * blockDim.x + threadIdx.x;
  const double mine = me < p.n_sites ? s[me] : 0.0;
  int rank = 0;
  for (int t0 = 0; t0 < p.n_sites; t0 += 256) {
    const int q = t0 + threadIdx.x;
    tile[threadIdx.x] = q < p.n_sites ? s[q] : -1.0;
    __syncthreads();
    const int lim = min(256, p.n_sites - t0);
    for (int k = 0; k < lim; k++) {
      const double v = tile[k];
      rank += (v > mine) || (v == mine && (t0 + k) < me);
    }
    __syncthreads();
  }
  if (me < p.n_sites) {
    const int mi = me / p.grid_n;
    p.order[base + rank] = (uint16_t)((mi << 8) | (me - mi * p.grid_n));  // packed (i, j) of the site
    const double pre = p.prefix[((size_t)c_pc_rclass[pc] * EG_NY + y) * p.n_sites + me];
    p.walk[base + rank] = make_double2(mine, pre);
  }
}

}  // namespace

cudaError_t eg_build_site_tables(const EgSiteBuildParams& p, cudaStream_t stream, int* launches) {
  dim3 g1((p.n_sites + 127) / 128, EG_NY, 1);
  eg_site_prefix_kernel<<<g1, 128, 0, stream>>>(p);
  dim3 g2((p.n_sites + 127) / 128, EG_NY, EG_N_PCLASS);
  eg_site_static_kernel<<<g2, 128, 0, stream>>>(p);
  dim3 g3((p.n_sites + 255) / 256, EG_NY, EG_N_PCLASS);
  eg_site_rank_kernel<<<g3, 256, 0, stream>>>(p);
  if (launches) *launches = 3;
  return cudaGetLastError();
}
