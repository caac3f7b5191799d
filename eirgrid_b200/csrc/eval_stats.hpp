// eval_stats.hpp — merging of eg_eval_stats records, one definition for the device fold (evaluate.cu) and the host merge
// (eg_eval_stats_merge): both compile this code without contraction (--fmad=false, -ffp-contract=off), so they give the same bits.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include "../../include/eirgrid_b200.h"

#ifdef __CUDACC__
#define EG_EVAL_HD __host__ __device__
#else
#define EG_EVAL_HD
#endif

namespace egeval {

constexpr int kMoments = EG_EVAL_N_FINAL + EG_N_YEARS * EG_EVAL_N_YEAR_FIELDS;  // moment entries: final metrics, then yearly

static_assert(offsetof(eg_eval_stats, yearly) == offsetof(eg_eval_stats, final_metrics) + EG_EVAL_N_FINAL * sizeof(eg_moments),
              "the moment entries are indexed as one array");
static_assert(sizeof(eg_eval_stats) - offsetof(eg_eval_stats, n_flagged) == EG_EVAL_COUNTER_WORDS * sizeof(uint64_t),
              "the counters run from n_flagged to the end of the record");

EG_EVAL_HD inline eg_moments* moments(eg_eval_stats* s) { return s->final_metrics; }
EG_EVAL_HD inline const eg_moments* moments(const eg_eval_stats* s) { return s->final_metrics; }
EG_EVAL_HD inline uint64_t* counters(eg_eval_stats* s) { return &s->n_flagged; }
EG_EVAL_HD inline const uint64_t* counters(const eg_eval_stats* s) { return &s->n_flagged; }

// x takes the place of the current maximum (minimum): larger (smaller), or the current one is NaN and x is not. NaN values are
// thus passed over unless every value is NaN.
EG_EVAL_HD inline bool above(double cur, double x) { return x > cur || (cur != cur && x == x); }
EG_EVAL_HD inline bool below(double cur, double x) { return x < cur || (cur != cur && x == x); }
EG_EVAL_HD inline bool same(double a, double b) { return a == b || (a != a && b != b); }

// a <- a (na values) followed by b (nb values): Chan, Golub and LeVeque's pairwise update of the mean and the sum of squared
// deviations. An empty side leaves the other one unchanged, bit for bit.
EG_EVAL_HD inline void merge_moments(eg_moments& a, uint64_t na, const eg_moments& b, uint64_t nb) {
  if (nb == 0) return;
  if (na == 0) { a = b; return; }
  const double fa = (double)na, fb = (double)nb, n = fa + fb;
  const double d = b.mean - a.mean;
  a.mean = a.mean + d * (fb / n);
  a.m2 = a.m2 + b.m2 + d * d * (fa * fb / n);
  if (below(a.min, b.min)) a.min = b.min;
  if (above(a.max, b.max)) a.max = b.max;
}

// the best / worst episode ids of a followed by b, from the score moments of both BEFORE they are merged; among equal scores
// the lower id is kept
EG_EVAL_HD inline void merge_extreme_ids(uint64_t& best_a, uint64_t& worst_a, const eg_moments& score_a, uint64_t na, uint64_t best_b,
                                         uint64_t worst_b, const eg_moments& score_b, uint64_t nb) {
  if (nb == 0) return;
  if (na == 0) { best_a = best_b; worst_a = worst_b; return; }
  if (above(score_a.max, score_b.max)) best_a = best_b;
  else if (same(score_a.max, score_b.max) && best_b < best_a) best_a = best_b;
  if (below(score_a.min, score_b.min)) worst_a = worst_b;
  else if (same(score_a.min, score_b.min) && worst_b < worst_a) worst_a = worst_b;
}

}  // namespace egeval
