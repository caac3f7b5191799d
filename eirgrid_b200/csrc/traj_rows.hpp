// traj_rows.hpp — how an action record (eg_traj) is read, ONE source for the host and the device: where each year's row lies,
// which counts are cut at the capacity, and the lists the update rule sees in a row (quirk Q10). The host rule
// (weights.cpp), the device rule (update.cu), the batch statistics (stats.cu), the evaluation (evaluate.cu) and the CSV export
// (report_files.cpp) read records through these functions only.
#pragma once
#include "tables.h"

#if defined(__CUDACC__)
#define EG_TRAJ_HD __host__ __device__ __forceinline__
#define EG_TRAJ_ANY_CALLABLE _Pragma("nv_exec_check_disable")  // the host rule passes host lambdas
#else
#define EG_TRAJ_HD inline
#define EG_TRAJ_ANY_CALLABLE
#endif

// One year's row: its first slot, then the deficit actions, then the additional actions.
struct EgTrajRow {
  int row, nd, na;
};

// The row that starts after `start` slots with nd deficit and na additional actions. Rows are stored back to back; counts that
// run past the capacity (never written by the episode kernels) are cut, so a row never reads past the record.
EG_TRAJ_HD EgTrajRow eg_traj_row_at(int start, int nd, int na) {
  const int row = start < EG_TRAJ_CAPACITY ? start : EG_TRAJ_CAPACITY;
  nd = nd < EG_TRAJ_CAPACITY - row ? nd : EG_TRAJ_CAPACITY - row;
  na = na < EG_TRAJ_CAPACITY - row - nd ? na : EG_TRAJ_CAPACITY - row - nd;
  return {row, nd, na};
}

// Year y's row, given year y - 1's (EgTrajRow{} before the first year): the sequential form.
EG_TRAJ_HD EgTrajRow eg_traj_next_row(const eg_traj& t, int y, const EgTrajRow& prev) {
  return eg_traj_row_at(prev.row + prev.nd + prev.na, t.n_deficit[y], t.n_additional[y]);
}

// The lists a row puts into the shared weights (transfer_recorded_actions_from, strategy.rs:313-342): the run list is the
// deficit actions followed by the additional actions, the deficit list the deficit actions. Replay iterations record every
// additional action twice and the first four deficit actions twice in the deficit list (sampling.rs:97-99,262-264 +
// simulation.rs:197,406-409; quirk Q10). Codes that are not action codes never come from the device; they are skipped, so a
// malformed record cannot index the tables with them.
EG_TRAJ_ANY_CALLABLE
template <typename F>
EG_TRAJ_HD void eg_for_each_run(const uint8_t* a, int nd, int na, bool replay, F&& f) {
  for (int i = 0; i < nd; i++) {
    const int c = a[i];
    if (c < EG_N_ACTIONS) f(c);
  }
  for (int i = nd; i < nd + na; i++) {
    const int c = a[i];
    if (c < EG_N_ACTIONS) {
      f(c);
      if (replay) f(c);
    }
  }
}
EG_TRAJ_ANY_CALLABLE
template <typename F>
EG_TRAJ_HD void eg_for_each_deficit(const uint8_t* a, int nd, bool replay, F&& f) {
  for (int i = 0; i < nd; i++) {
    const int c = a[i];
    if (c < EG_N_ACTIONS) {
      f(c);
      if (replay && i < 4) f(c);
    }
  }
}

#if defined(__CUDACC__)
// The warp form: lane y < EG_NY gets year y's row from one shuffle scan over the counts, the other lanes an empty row.
// All 32 lanes must call this together.
__device__ __forceinline__ EgTrajRow eg_warp_traj_row(const eg_traj* t, int lane) {
  int nd = 0, na = 0;
  if (lane < EG_NY) { nd = t->n_deficit[lane]; na = t->n_additional[lane]; }
  int end = nd + na;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xFFFFFFFFu, end, o);
    if (lane >= o) end += v;
  }
  return eg_traj_row_at(end - (nd + na), nd, na);
}

// One warp walks the items of one record: year after year, current_run_actions (the whole row: deficit actions, then
// additional actions) followed by current_deficit_actions (the row's deficit part again), ~40 items in all, most of them in
// 2025. The items are numbered through all years (warp prefix sum) and dealt out 32 at a time, each lane finding its item's
// year by binary search over the prefix sums. visit(y, i, nrun, nd, a) is called for item i of year y with action code a:
// i < nrun is slot i of the row, i >= nrun is deficit action i - nrun; nd is the year's deficit count. All 32 lanes must call
// this together.
template <typename Visit>
__device__ __forceinline__ void eg_warp_traj_items(const eg_traj* t, int lane, Visit&& visit) {
  const EgTrajRow r = eg_warp_traj_row(t, lane);
  const int row = r.row, nrun = r.nd + r.na, cnt = nrun + r.nd;
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
#endif
