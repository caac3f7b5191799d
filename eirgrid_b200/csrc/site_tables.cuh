// site_tables.cuh — GPU construction of the static candidate-site tables (site_tables.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct EgSiteBuildParams {
  int grid_n;
  int n_sites;
  double step;
  int n_settlements;
  const double* sx;        // [S]
  const double* sy;
  const uint32_t* pop;     // [26][S] population of each settlement in each year
  int n_existing;
  const double* ex;        // [E]
  const double* ey;
  int n_coast;
  const double* cx;        // [C]
  const double* cy;
  double size_factor;
  // outputs
  double* prefix;          // [6][26][n_sites]  score after settlements and existing plants per radius class
  double* coast_factor;    // [n_sites]
  double* site_opinion;    // [n_sites]
  double* static_unsorted; // [7][26][n_sites] scratch: static scores in site order
  uint16_t* order;         // [7][26][n_sites]
  double2* walk;           // [7][26][n_sites] (static score, prefix score) in `order`: one 16-byte read per walk entry
};

// launches 3 kernels on `stream`; returns the number of launches in *launches
cudaError_t eg_build_site_tables(const EgSiteBuildParams& p, cudaStream_t stream, int* launches);
