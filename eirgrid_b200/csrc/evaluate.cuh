// evaluate.cuh — reduction of rollout outputs into an eg_eval_stats record (evaluate.cu).
#pragma once
#include <cuda_runtime.h>
#include "eval_stats.hpp"
#include "tables.h"

#define EG_EVAL_SLICE 256  // episodes per block of the block pass (one thread each); fixed, so the partition depends on n only

struct EgEvalPartial {  // one block's slice: its moments and the global ids of its best and worst scores
  eg_moments m[egeval::kMoments];
  uint64_t best, worst;
};

struct EgEvalParams {
  const eg_result* results;
  const eg_traj* traj;
  const eg_yearly* yearly;         // nullable: no per-year part
  uint32_t n;                      // at most EG_EVAL_CHUNK
  unsigned long long first_global; // global id of episode 0
  eg_eval_stats* acc;              // device record the chunk is folded into
  EgEvalPartial* partials;         // [EG_EVAL_CHUNK / EG_EVAL_SLICE]
};

// 2 launches (none for n = 0): block pass (counters straight into acc, moments into the partials), then the fold of the
// partials into acc in block order
cudaError_t eg_launch_eval(const EgEvalParams& p, cudaStream_t stream);
