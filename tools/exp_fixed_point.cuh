// EXPERIMENT (not used by the library): fixed-point evaluation of the exponential for the swish / tanh / softmax fast
// paths -- 3 FP64 instructions per exponential instead of 7 (swish and tanh 7 instead of 12), accuracy 2.8e-14.
// Measured in k_fwd3 (profiles/r02_fwd3_v1_ncu.txt -> r02_fwd3_v2_ncu.txt): non-MMA FP64 instructions 1.38 G -> 0.84 G
// per launch, FP64 pipe 14.8 % -> 9.1 % busy, launch time 16.62 -> 16.64 ms: the 12 integer / FP32 instructions that
// replace 5 FP64 instructions cost as much (0.75 clk each against 2.9, tools/stream_mix.cu, tools/fp64_mix.cu), and the
// block-masked kernel (issue-bound) lost 3 %.  Kept here with its accuracy check (tools/exp_fix_check.cu) because the
// reduction itself is reusable; the library keeps the 4e-16 table + polynomial evaluation.
// The table must be pre-scaled: tab[j] = 2^(j/2048 - EXPFIX_TAB_BIAS).
#pragma once
#include "../npbnn_b200/csrc/bnn_common.cuh"
#define EXPFIX_TAB_BIAS 64
// ------------------------------------------------------------------------------------------------
// Fixed-point evaluation of the exponential (2048-entry table only) for the fast paths: 3 FP64 instructions.
//
// Every non-MMA FP64 instruction costs 2.5 clk of the FP64 pipe the DMMAs need, FP32 and 32-bit integer instructions
// 0.2 clk (tools/pipe_cost.cu; IMAD.HI / IMAD.WIDE cost 3.7 clk -- 64-bit integer products are no way out), and the
// table scheme above spends 7 FP64 instructions per exponential.  Here ONE FMA does the whole argument reduction
//     t = z * (SCALE * 2^11 / ln 2) + 1.5 * 2^18          |SCALE * z| < 2^17 ln2 / 2^11 = 44.36
// t lies in [2^18, 2^19), its unit in the last place is 2^-34: with u = the scaled argument, the low 20 bits of the
// high word hold 4 * (2^17 + floor(u)) + (the two leading fraction bits), the low word holds the next 32 fraction
// bits.  exp(SCALE z) = 2^(u / 2^11) = 2^n * tab[j] * D1 with j = floor(u) mod 2^11, n = floor(u) >> 11 and
//     D1 = 2^(f / 2^11) = 1 + c f + (c^2 f^2 / 2 + c^3 f^3 / 6),   c = ln2 / 2^11,  f = frac(u) in [0, 1).
// The bracket (< 5.8e-8) is evaluated in FP32 from the 23 leading bits of f and rounded to an integer g in units of
// c 2^-34 by the 2^23 trick; the 34 fraction bits plus g, placed under the exponent of 2^52, ARE the double
// 2^52 + (f + g) 2^34, and one FMA with c'' = Q 2^-98, K0 = 1 - Q 2^-46 (Q = round(c 2^64), 53 bits, so that both
// constants are exact and the 2^52 offset cancels exactly inside the FMA) gives D1.  2^n goes into the exponent of the
// pre-scaled table value with a mask and a shift-add.  The caller folds Ts * D1 into the FMA that forms 1 + exp.
// Accuracy: the rounding of t leaves f off by <= 2^-35, g by <= 0.6 units: exp is off by <= 2.2e-14 relative
// (rms 8e-15, unbiased; tools/exp_fix_check.cu) -- the log-likelihood by ~1e-14 relative against a tolerance of 1e-9.
// Arguments outside the range (and inf / NaN) take the callers' guarded path with the table scheme above.
// ------------------------------------------------------------------------------------------------
#define BNN_FIX_THR_1 0x40460000     // 44.0: |z| below it keeps exp(+-z) inside the fixed-point range
#define BNN_FIX_THR_2 0x40360000     // 22.0: the same for exp(2z)
template <int SCALE>
__device__ __forceinline__ void bnn_exp_split(double z, const double* __restrict__ tab, double& Ts, double& D1) {
  static_assert(BNN_EXP_TAB_BITS == 11, "fixed-point exponential: 2048-entry table");
  static_assert(SCALE == -1 || SCALE == 1 || SCALE == 2, "exp(-z), exp(z) or exp(2z)");
  const double t = fma(z, (double)SCALE * 2954.639443740597, 393216.0);
  const unsigned hi = (unsigned)__double2hiint(t), F = (unsigned)__double2loint(t);
  const double T = *reinterpret_cast<const double*>(reinterpret_cast<const char*>(tab) + ((hi << 1) & 0x3FF8u));
  Ts = __hiloint2double(__double2hiint(T) + (int)((hi & 0x000FE000u) << 7), __double2loint(T));
  // second-order terms in FP32: y = 1 + (23 leading bits of f); f re-centred on its truncation interval
  const float y = __uint_as_float((__funnelshift_r(F, hi, 11) & 0x007FFFFFu) | 0x3F800000u);
  const float ff = y - 0.99999994f;
  const float h = fmaf(327.98926f, ff, 2907270.0f);                  // 2^34 (c^2 / 2 + c^3 f / 6) / c
  const float gm = fmaf(ff * ff, h, 8388608.0f);                     // 2^23 + g
  const unsigned long long w = (((unsigned long long)(0x43300000u | (hi & 3u))) << 32 | F) +
                               (unsigned long long)(__float_as_uint(gm) - 0x4B000000u);
  D1 = fma(__longlong_as_double((long long)w), 1.9700427758378546e-14, -87.722839111673);
}

// Softmax terms of the likelihood epilogue, exp(x) for x <= 0, through the fixed-point evaluation: arguments below -44
// give 0, i.e. a term below 8e-20 of a sum that is >= 1 -- less than half a unit in the last place of the sum
// (NaN propagates).  Only the SUM is used in likelihood mode (the -inf of an underflowing log-softmax is decided on z_y - max, not on this value);
// prediction mode reports the individual terms and keeps bnn_exp_neg.
__device__ __forceinline__ double bnn_exp_neg_fast(double x, const double* __restrict__ tab) {
  const int hx = __double2hiint(x);
  const bool big = (hx & 0x7fffffff) >= BNN_FIX_THR_1;                // also inf / NaN
  double Ts, D1;
  bnn_exp_split<1>(__hiloint2double(big ? 0 : hx, big ? 0 : __double2loint(x)), tab, Ts, D1);
  double res = Ts * D1;
  res = big ? 0.0 : res;
  const bool is_nan = bnn_is_nan_int(x);
  return __hiloint2double(__double2hiint(res) | (is_nan ? 0x7ff80000 : 0), __double2loint(res));
}


template <int ACT>
__device__ __forceinline__ bool expfix_needs_care(double z) {
  return (__double2hiint(z) & 0x7fffffff) >= (ACT == BNN_ACT_SWISH ? BNN_FIX_THR_1 : BNN_FIX_THR_2);
}
template <int ACT>
__device__ __forceinline__ double expfix_act_fast(double z, const double* __restrict__ tab) {
  double Ts, D1;
  bnn_exp_split<(ACT == BNN_ACT_SWISH) ? -1 : 2>(z, tab, Ts, D1);
  const double y = bnn_rcp(fma(Ts, D1, 1.0));
  return (ACT == BNN_ACT_SWISH) ? z * y : fma(-2.0, y, 1.0);
}
