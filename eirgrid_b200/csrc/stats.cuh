// stats.cuh — batch-synchronous update statistics (stats.cu).
#pragma once
#include <cuda_runtime.h>
#include "tables.h"
#include "weights.hpp"

struct EgStatsParams {
  EgContrastConsts consts;
  const EgPolicyDevice* policy;   // snapshot the batch was sampled from (best lists)
  const eg_result* results;
  const eg_traj* trajs;
  uint32_t n;
  int64_t* stats;                 // [EG_STATS_WORDS], accumulated
  double* best_score;             // [1]
  unsigned long long* best_index; // [1]
  double ln100;
};

// The winner record of a shard: its best score and the episode that holds it. One flat record of EG_BEST_RECORD_BYTES
// without padding, so that ranks can exchange it as raw bytes (int64 words).
struct EgBestRecord {
  double score;
  int64_t episode;  // global id
  eg_result result;
  eg_traj traj;
};
static_assert(sizeof(EgBestRecord) == EG_BEST_RECORD_BYTES &&
                  sizeof(EgBestRecord) == sizeof(double) + sizeof(int64_t) + sizeof(eg_result) + sizeof(eg_traj),
              "the winner record is EG_BEST_RECORD_BYTES without padding");
static_assert(sizeof(EgBestRecord) % 8 == 0 && alignof(EgBestRecord) == 8, "the winner record is packed and exchanged in 64-bit words");

// 1 launch: the winner record (EgBestRecord) of the shard's best episode; `record` is 8-byte aligned
cudaError_t eg_launch_pack_best(const eg_result* results, const eg_traj* trajs, uint32_t n, const double* best_score,
                                const unsigned long long* best_index, unsigned long long first_global, void* record, cudaStream_t stream);

// 3 launches: reset of the best slot, accumulation + max score, lowest index holding the max
cudaError_t eg_launch_stats(const EgStatsParams& p, cudaStream_t stream);
