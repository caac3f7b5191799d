// traj_items.cuh — one warp walks the items of one episode's action record (eg_traj); shared by stats.cu and evaluate.cu.
#pragma once
#include "tables.h"

// The record's items are, year after year, current_run_actions (the whole row: deficit actions, then additional actions)
// followed by current_deficit_actions (the row's deficit part again), ~40 items in all, most of them in 2025. Lane y holds
// year y's counts; the items are numbered through all years (warp prefix sum) and dealt out 32 at a time, each lane finding
// its item's year by binary search over the prefix sums. Counts that run past the capacity (never written by the episode
// kernels) are cut. visit(y, i, nrun, nd, a) is called for item i of year y with action code a: i < nrun is slot i of the
// row, i >= nrun is deficit action i - nrun; nd is the year's deficit count. All 32 lanes must call this together.
template <typename Visit>
__device__ __forceinline__ void eg_warp_traj_items(const eg_traj* t, int lane, Visit&& visit) {
  int nd = 0, nrun = 0;
  if (lane < EG_NY) { nd = t->n_deficit[lane]; nrun = nd + t->n_additional[lane]; }
  // first slot of each year's row in the record (rows are stored back to back)
  int row_end = nrun;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xFFFFFFFFu, row_end, o);
    if (lane >= o) row_end += v;
  }
  int row = row_end - nrun;
  if (row > EG_TRAJ_CAPACITY) row = EG_TRAJ_CAPACITY;
  if (row + nrun > EG_TRAJ_CAPACITY) { nrun = EG_TRAJ_CAPACITY - row; nd = min(nd, nrun); }
  const int cnt = nrun + nd;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
    if (lane >= o) incl += v;
  }
  const int total = __shfl_sync(0xFFFFFFFFu, incl, 31);
  for (int base = 0; base < total; base += 32) {
    const int q = base + lane;
    int y = 0;  // number of years whose items all come before item q
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
      const int v = __shfl_sync(0xFFFFFFFFu, incl, y + step - 1);
      if (v <= q) y += step;
    }
    const int y_incl = __shfl_sync(0xFFFFFFFFu, incl, y), y_cnt = __shfl_sync(0xFFFFFFFFu, cnt, y);
    const int y_nrun = __shfl_sync(0xFFFFFFFFu, nrun, y), y_row = __shfl_sync(0xFFFFFFFFu, row, y);
    if (q >= total) continue;
    const int i = q - (y_incl - y_cnt);
    const int a = t->actions[y_row + (i < y_nrun ? i : i - y_nrun)];
    visit(y, i, y_nrun, y_cnt - y_nrun, a);
  }
}
