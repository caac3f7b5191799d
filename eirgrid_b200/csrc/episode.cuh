// episode.cuh — launch interface of the episode kernels (episode.cu).
#pragma once
#include <cuda_runtime.h>
#include "tables.h"

struct EgEpisodeParams {
  EgDeviceMap map;
  const EgPolicyDevice* policy;  // rollout mode (device pointer)
  const eg_traj* replay_in;      // trajectory-replay mode (device pointer)
  eg_result* out;
  eg_traj* traj;                 // nullable
  eg_sites* sites;               // nullable
  eg_yearly* yearly;             // nullable
  int nf_entries;                // size of the compact distance/radius table copied to shared memory (narrow maps)
  uint32_t* next_episode;        // device counter the persistent warps claim episodes from (zeroed by the launcher)
  unsigned long long seed;
  unsigned long long first_episode;
  uint32_t n;
  uint32_t cost_only;
  uint32_t energy_sales;
  uint32_t same_stream;
  uint32_t replay_best;
  uint32_t stagnation;           // host copy of EgPolicyDevice::iwi > 500 (which sampler the lean instantiation carries)
  uint32_t count_weights;        // the uploaded policy has action-count weights (host copy of EgPolicyDevice::has_count_weights)
  double ln100;                  // ln(MAX_ACCEPTABLE_COST*100/MAX_ACCEPTABLE_COST), host libm (scoring.rs:13,32)
};

cudaError_t eg_launch_rollout(const EgEpisodeParams& p, cudaStream_t stream);
cudaError_t eg_launch_replay(const EgEpisodeParams& p, cudaStream_t stream);
