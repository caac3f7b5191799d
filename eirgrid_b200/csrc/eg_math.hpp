// eg_math.hpp — exp / ln / pow for the weight-update rule and Philox4x32-10, ONE source for the host and the device.
//
// The reference's update (ai/learning/weights/learning.rs:131-373) calls f64::exp, f64::powf and (through score_metrics,
// ai/metrics/scoring.rs:12-13) f64::ln with per-episode arguments: the deterioration of every episode goes through
// powf(0.3), the stagnation counter through exp(-iwi/500) and powf(1.8). Rust forwards these to the platform libm, so the
// reference itself gives last-bit-different weights on glibc, musl and macOS. For the device form of the update
// (update.cu) to end with the SAME table as the host form (weights.cpp) the two must round identically, which no pair of
// vendor libms does (CUDA's pow is within 1-2 ulp of glibc's, not equal to it).
//
// These functions are built from IEEE + - * / and explicit fma only (double-double arithmetic, ~100 bits), so host
// (-ffp-contract=off) and device (--fmad=false) execute the same operations and return the same bits. Their results are the
// correctly rounded values except when the exact result lies within ~2^-45 ulp of a rounding boundary (never observed;
// tests/test_eg_math.py checks 10^5 arguments per function against 60-digit decimal arithmetic); glibc's own functions are
// within 1 ulp and agree with these on > 99.9 % of the arguments the rule produces (same test), which is what bounds the
// distance to the CPU oracle (glibc): a last-bit difference in a rare factor, never a different branch.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define EGM_HD __host__ __device__ inline
#else
#define EGM_HD inline
#endif

namespace egm {

struct dd {  // value = hi + lo, |lo| <= ulp(hi)/2
  double hi, lo;
};

EGM_HD dd two_sum(double a, double b) {
  const double s = a + b, bb = s - a;
  return {s, (a - (s - bb)) + (b - bb)};
}
EGM_HD dd quick_two_sum(double a, double b) {  // |a| >= |b|
  const double s = a + b;
  return {s, b - (s - a)};
}
EGM_HD dd two_prod(double a, double b) {
  const double p = a * b;
  return {p, fma(a, b, -p)};
}
EGM_HD dd add(dd a, dd b) {
  dd s = two_sum(a.hi, b.hi);
  const dd t = two_sum(a.lo, b.lo);
  s.lo += t.hi;
  s = quick_two_sum(s.hi, s.lo);
  s.lo += t.lo;
  return quick_two_sum(s.hi, s.lo);
}
EGM_HD dd add_d(dd a, double b) {
  dd s = two_sum(a.hi, b);
  s.lo += a.lo;
  return quick_two_sum(s.hi, s.lo);
}
EGM_HD dd mul(dd a, dd b) {
  dd p = two_prod(a.hi, b.hi);
  p.lo += a.hi * b.lo + a.lo * b.hi;
  return quick_two_sum(p.hi, p.lo);
}
EGM_HD dd mul_d(dd a, double b) {
  dd p = two_prod(a.hi, b);
  p.lo += a.lo * b;
  return quick_two_sum(p.hi, p.lo);
}
EGM_HD dd neg(dd a) { return {-a.hi, -a.lo}; }

EGM_HD double from_bits(uint64_t u) {
  double d;
  memcpy(&d, &u, sizeof(d));
  return d;
}
EGM_HD uint64_t to_bits(double d) {
  uint64_t u;
  memcpy(&u, &d, sizeof(u));
  return u;
}
EGM_HD double pow2(int k) { return from_bits((uint64_t)(k + 1023) << 52); }  // -1022 <= k <= 1023
EGM_HD double scale2(double v, int k) {  // v * 2^k, stepwise so that the scale factors stay normal
  while (k > 1000) { v *= pow2(1000); k -= 1000; }
  while (k < -1000) { v *= pow2(-1000); k += 1000; }
  return v * pow2(k);
}

// ln 2 and the series coefficients as double-doubles (generated with 80-digit decimal arithmetic)
EGM_HD dd ln2() { return {0x1.62e42fefa39efp-1, 0x1.abc9e3b39803fp-56}; }
EGM_HD dd inv_odd(int k) {  // 1 / (2k + 1), k = 0..22
  switch (k) {
    case 0: return {0x1.0000000000000p+0, 0x0.0p+0};
    case 1: return {0x1.5555555555555p-2, 0x1.5555555555555p-56};
    case 2: return {0x1.999999999999ap-3, -0x1.999999999999ap-57};
    case 3: return {0x1.2492492492492p-3, 0x1.2492492492492p-57};
    case 4: return {0x1.c71c71c71c71cp-4, 0x1.c71c71c71c71cp-58};
    case 5: return {0x1.745d1745d1746p-4, -0x1.745d1745d1746p-59};
    case 6: return {0x1.3b13b13b13b14p-4, -0x1.3b13b13b13b14p-58};
    case 7: return {0x1.1111111111111p-4, 0x1.1111111111111p-60};
    case 8: return {0x1.e1e1e1e1e1e1ep-5, 0x1.e1e1e1e1e1e1ep-61};
    case 9: return {0x1.af286bca1af28p-5, 0x1.af286bca1af28p-59};
    case 10: return {0x1.8618618618618p-5, 0x1.8618618618618p-59};
    case 11: return {0x1.642c8590b2164p-5, 0x1.642c8590b2164p-60};
    case 12: return {0x1.47ae147ae147bp-5, -0x1.eb851eb851eb8p-61};
    case 13: return {0x1.2f684bda12f68p-5, 0x1.2f684bda12f68p-59};
    case 14: return {0x1.1a7b9611a7b96p-5, 0x1.1a7b9611a7b96p-61};
    case 15: return {0x1.0842108421084p-5, 0x1.0842108421084p-60};
    case 16: return {0x1.f07c1f07c1f08p-6, -0x1.f07c1f07c1f08p-61};
    case 17: return {0x1.d41d41d41d41dp-6, 0x1.0750750750750p-60};
    case 18: return {0x1.bacf914c1bad0p-6, -0x1.bacf914c1bad0p-60};
    case 19: return {0x1.a41a41a41a41ap-6, 0x1.0690690690690p-60};
    case 20: return {0x1.8f9c18f9c18fap-6, -0x1.f3831f3831f38p-61};
    case 21: return {0x1.7d05f417d05f4p-6, 0x1.7d05f417d05f4p-62};
    default: return {0x1.6c16c16c16c17p-6, -0x1.f49f49f49f49fp-61};
  }
}
EGM_HD dd inv_fact(int j) {  // 1 / j!, j = 1..13
  switch (j) {
    case 1: return {0x1.0000000000000p+0, 0x0.0p+0};
    case 2: return {0x1.0000000000000p-1, 0x0.0p+0};
    case 3: return {0x1.5555555555555p-3, 0x1.5555555555555p-57};
    case 4: return {0x1.5555555555555p-5, 0x1.5555555555555p-59};
    case 5: return {0x1.1111111111111p-7, 0x1.1111111111111p-63};
    case 6: return {0x1.6c16c16c16c17p-10, -0x1.f49f49f49f49fp-65};
    case 7: return {0x1.a01a01a01a01ap-13, 0x1.a01a01a01a01ap-73};
    case 8: return {0x1.a01a01a01a01ap-16, 0x1.a01a01a01a01ap-76};
    case 9: return {0x1.71de3a556c734p-19, -0x1.c154f8ddc6c00p-73};
    case 10: return {0x1.27e4fb7789f5cp-22, 0x1.cbbc05b4fa99ap-76};
    case 11: return {0x1.ae64567f544e4p-26, -0x1.c062e06d1f209p-80};
    case 12: return {0x1.1eed8eff8d898p-29, -0x1.2aec959e14c06p-83};
    default: return {0x1.6124613a86d09p-33, 0x1.f28e0cc748ebep-87};
  }
}

// ln(x) as a double-double, x positive and finite.
// x = m * 2^e with m in (sqrt(1/2), sqrt 2]; ln m = 2 atanh(s), s = (m - 1) / (m + 1), |s| <= 0.1716;
// atanh(s) = s * sum_k s^(2k) / (2k + 1), 23 terms (the first omitted term is below 2^-118).
EGM_HD dd log_dd(double x) {
  int e = 0;
  if (x < 0x1p-1022) {  // subnormal
    x *= 0x1p54;
    e = -54;
  }
  const uint64_t bits = to_bits(x);
  e += (int)((bits >> 52) & 0x7FF) - 1023;
  double m = from_bits((bits & 0x000FFFFFFFFFFFFFull) | 0x3FF0000000000000ull);  // [1, 2)
  if (m > 0x1.6a09e667f3bcdp+0) {
    m *= 0.5;
    e += 1;
  }
  const double num = m - 1.0;           // exact
  const dd den = two_sum(m, 1.0);       // exact
  // s = num / den to double-double accuracy: two steps of long division
  const double q1 = num / den.hi;
  const dd p = two_prod(q1, den.hi);
  const double r = ((num - p.hi) - p.lo) - q1 * den.lo;
  const double q2 = r / den.hi;
  const dd s = quick_two_sum(q1, q2);
  const dd s2 = mul(s, s);
  dd sum = inv_odd(22);
  for (int k = 21; k >= 0; k--) sum = add(mul(sum, s2), inv_odd(k));
  dd lm = mul(s, sum);
  lm.hi *= 2.0;
  lm.lo *= 2.0;
  if (e == 0) return lm;
  return add(mul_d(ln2(), (double)e), lm);
}

// exp(a) for a double-double argument, rounded to double.
// a = k ln 2 + r, |r| <= 0.35; exp(r) - 1 from the Taylor series of r / 64 (13 terms) and six doublings
// (1 + p)^2 - 1 = 2p + p^2.
EGM_HD double exp_dd(dd a) {
  if (a.hi != a.hi) return a.hi;
  if (a.hi > 709.782712893384) return from_bits(0x7FF0000000000000ull);
  if (a.hi < -745.2) return 0.0;
  const double kd = rint(a.hi * 0x1.71547652b82fep+0);
  dd r = add(a, neg(mul_d(ln2(), kd)));
  r.hi *= 0x1p-6;
  r.lo *= 0x1p-6;
  dd s = inv_fact(13);
  for (int j = 12; j >= 1; j--) s = add(mul(s, r), inv_fact(j));
  dd p = mul(s, r);
  for (int i = 0; i < 6; i++) {
    dd twice = p;
    twice.hi *= 2.0;
    twice.lo *= 2.0;
    p = add(twice, mul(p, p));
  }
  const dd v = add_d(p, 1.0);
  return scale2(v.hi, (int)kd);
}

EGM_HD double exp(double a) { return exp_dd({a, 0.0}); }

EGM_HD double log(double x) {
  if (x != x) return x;
  if (x < 0.0) return from_bits(0x7FF8000000000000ull);
  if (x == 0.0) return from_bits(0xFFF0000000000000ull);
  if (x == from_bits(0x7FF0000000000000ull)) return x;
  if (x == 1.0) return 0.0;
  return log_dd(x).hi;
}

// pow(x, y) for the arguments the update rule produces (finite y; x of any sign): NaN for a negative base with a
// non-integer exponent like libm (quirk Q9 rests on it), exact for the trivial cases.
EGM_HD double pow(double x, double y) {
  if (y == 0.0 || x == 1.0) return 1.0;
  if (x != x || y != y) return from_bits(0x7FF8000000000000ull);
  const double inf = from_bits(0x7FF0000000000000ull);
  double sign = 1.0;
  if (x < 0.0) {
    if (y != rint(y)) return from_bits(0x7FF8000000000000ull);
    if (fabs(y) < 0x1p53 && fmod(fabs(y), 2.0) == 1.0) sign = -1.0;
    x = -x;
  }
  if (x == 0.0) return y > 0.0 ? 0.0 * sign : inf * sign;
  if (x == inf) return y > 0.0 ? inf * sign : 0.0 * sign;
  if (y == 1.0) return sign * x;
  return sign * exp_dd(mul_d(log_dd(x), y));
}

// Philox4x32-10 (Salmon et al., SC '11) of the counter x under the key (k0, k1), in place: every counter-based stream
// outside the episode kernel (whose philox_u64 is its own, tuned form) draws from this one
EGM_HD void philox4x32_10(uint32_t x[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; r++) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * x[0], p1 = (uint64_t)0xCD9E8D57u * x[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ x[1] ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ x[3] ^ k1, n3 = (uint32_t)p0;
    x[0] = n0; x[1] = n1; x[2] = n2; x[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

// the low 64 bits of a Philox output, words (lo, hi), as a 53-bit uniform in [0, 1)
EGM_HD double uniform53(uint32_t lo, uint32_t hi) { return (double)((((uint64_t)hi << 32) | lo) >> 11) * (1.0 / 9007199254740992.0); }

}  // namespace egm
