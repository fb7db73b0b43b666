// lfr_math.cuh — per-edge arithmetic of the multi-view refinement cost, fp64.
//
//   eval_edge()         cost.cc:13-48 (biquadratic interpolation with clamping)
//                       + cost.cc:78-90 (residual x2 - x1 - flow(x1))
//                       + Ceres loss (ScaledLoss(Cauchy|Tukey), SURVEY A.2)
//   ls_next_step()      Ceres ArmijoLineSearch step-size selection by cubic /
//                       quintic Hermite interpolation (SURVEY A.6, polynomial.cc)
//
// The flow grid is read as five 128-bit words (the 80-byte lfr_edge record) and
// widened to fp64 in registers; no tensor cores: this is 2-DoF sparse NLLS.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/lfr.h"

namespace lfr {

struct DevConsts {
  double bound;
  double cauchy_b, cauchy_c;          // a^2, 1/a^2
  double tukey_a2, tukey_inv_a2;      // a^2, 1/a^2
  double tukey_rho0, tukey_rho1;      // a^2/6 & 0.5 (Ceres 1.x)  or  a^2/3 & 1.0 (2.x)
  double f_tol, g_tol, p_tol;
  double radius0, radius_max, radius_min;
  double min_rel_decrease, min_diag, max_diag;
  double ls_suff, ls_max_contraction, ls_min_contraction, ls_min_step;
  int max_iter, max_invalid, max_ls_iter, linear_solver;
};

// Result of one residual-block evaluation, already in the form the assembly
// needs:  a = sim * rho'(|r|^2)  (Corrector: J~ = sqrt(a) J, r~ = sqrt(a) r),
// r = raw residual, M = I + grad(flow)  (so d r/d x_src = -M, d r/d x_dst = I).
struct EdgeEval {
  double a, r0, r1, m00, m01, m10, m11, half_rho;
};

__device__ __forceinline__ void lagrange3(double t, double L[3], double dL[3]) {
  // cost.cc:20-23, nodes at -0.5, 0, +0.5
  L[0] = 2. * t * (t - .5);
  L[1] = (-4.) * (t - .5) * (t + .5);
  L[2] = 2. * t * (t + .5);
  dL[0] = 4. * t - 1.;
  dL[1] = -8. * t;
  dL[2] = 4. * t + 1.;
}

// Scaled loss {0.5*rho, rho'} at s = |r|^2.
__device__ __forceinline__ void scaled_loss(int kind, double sim, double s, const DevConsts& K,
                                            double* half_rho, double* rho1) {
  if (kind == LFR_EDGE_CAUCHY) {
    const double sum = 1.0 + s * K.cauchy_c;
    *half_rho = 0.5 * sim * (K.cauchy_b * log(sum));
    *rho1 = sim * fmax(2.2250738585072014e-308, 1.0 / sum);
  } else {
    if (s <= K.tukey_a2) {
      const double v = 1.0 - s * K.tukey_inv_a2;
      const double v2 = v * v;
      *half_rho = 0.5 * sim * (K.tukey_rho0 * (1.0 - v2 * v));
      *rho1 = sim * (K.tukey_rho1 * v2);
    } else {
      *half_rho = 0.5 * sim * K.tukey_rho0;
      *rho1 = 0.0;
    }
  }
}

// q[0..4] = the 80-byte edge record as five float4 (q[4].z = sim, q[4].w = dst).
__device__ __forceinline__ EdgeEval eval_edge(const float4 q[5], int kind, double x1r, double x1c,
                                              double x2r, double x2c, const DevConsts& K) {
  const double row = fmax(fmin(x1r, .5), -.5);   // cost.cc:17-18
  const double col = fmax(fmin(x1c, .5), -.5);
  const bool row_free = (row == x1r), col_free = (col == x1c);  // cost.cc:38,41
  double Lr[3], dLr[3], Lc[3], dLc[3];
  lagrange3(row, Lr, dLr);
  lagrange3(col, Lc, dLc);
  // D[i][j][k] = flow[2*(3i+j)+k]
  const double D[3][3][2] = {
      {{(double)q[0].x, (double)q[0].y}, {(double)q[0].z, (double)q[0].w}, {(double)q[1].x, (double)q[1].y}},
      {{(double)q[1].z, (double)q[1].w}, {(double)q[2].x, (double)q[2].y}, {(double)q[2].z, (double)q[2].w}},
      {{(double)q[3].x, (double)q[3].y}, {(double)q[3].z, (double)q[3].w}, {(double)q[4].x, (double)q[4].y}}};
  double f[2], fr[2], fc[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    double v = 0., vr = 0., vc = 0.;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double t = Lc[0] * D[i][0][k] + Lc[1] * D[i][1][k] + Lc[2] * D[i][2][k];
      const double tc = dLc[0] * D[i][0][k] + dLc[1] * D[i][1][k] + dLc[2] * D[i][2][k];
      v += Lr[i] * t;
      vr += dLr[i] * t;
      vc += Lr[i] * tc;
    }
    f[k] = v;
    fr[k] = row_free ? vr : 0.;
    fc[k] = col_free ? vc : 0.;
  }
  EdgeEval o;
  o.r0 = x2r - x1r - f[0];   // cost.cc:87
  o.r1 = x2c - x1c - f[1];
  o.m00 = 1. + fr[0];
  o.m01 = fc[0];
  o.m10 = fr[1];
  o.m11 = 1. + fc[1];
  scaled_loss(kind, (double)q[4].z, o.r0 * o.r0 + o.r1 * o.r1, K, &o.half_rho, &o.a);
  return o;
}

// ---------------------------------------------------------------------------
// Line-search step selection (Ceres ArmijoLineSearch, polynomial.cc).
//
// Ceres fits the polynomial interpolating {value, gradient} at step 0, at the
// current trial step and (from the second contraction on) at the previous one,
// and takes the minimiser over [1e-3, 0.6] x current among: interval middle,
// interval ends, real parts of all roots of p', and the sample abscissae.  The
// same interpolant is built here in the normalised variable t = x / h
// (h = largest sample step), where the two constraints at 0 fix the two lowest
// coefficients and the rest is a 2x2 (cubic) or 4x4 (quintic) system — the same
// polynomial as Ceres' 4x4 / 6x6 Vandermonde solve, better conditioned (closed
// forms: a 2x2 solve, or the divided differences of the reduced cubic).  Only
// the real critical points inside the interval can win the minimisation, and
// those are bracketed exactly (see real_roots_in).  oracle/lfr_oracle.cc
// mirrors this operation for operation; quartic_roots_grid below is the
// lane-parallel route to the same quartic roots (the recursion is its fallback).
// ---------------------------------------------------------------------------
struct LsSample {
  double x, value, gradient;
  bool value_valid, gradient_valid;
};

__device__ __forceinline__ double poly_eval(const double* p, int n, double x) {
  double v = 0.0;
  for (int i = 0; i < n; ++i) v = v * x + p[i];
  return v;
}

// ---- real roots of a polynomial inside an interval ---------------------------
// MinimizePolynomial looks at the real parts of ALL roots of p', but a candidate
// only wins if its value is strictly below the best of {middle, ends}; on an
// interval the minimum of p is attained at an end or at a REAL critical point
// inside it, so complex roots and roots outside [lo, hi] can never be selected.
// The real roots inside the interval are found exactly and cheaply by
// recursion on the derivative: between two consecutive critical points a
// polynomial is monotone, so every sign change brackets exactly one root, which
// a safeguarded Newton iteration (Numerical Recipes' rtsafe) then polishes.
__device__ __forceinline__ void horner2(const double* q, int nq, double x, double* f, double* df) {
  double v = q[0], d = 0.0;
  for (int i = 1; i < nq; ++i) {
    d = d * x + v;
    v = v * x + q[i];
  }
  *f = v;
  *df = d;
}

// f / df for the Newton step: the correctly rounded single-precision reciprocal
// of df (MUFU.RCP + fix-up, bit-identical to the oracle's 1.0f / (float)df) is
// accurate enough to keep the quadratic convergence and replaces the double
// division, the longest dependent chain of the iteration.
__device__ __forceinline__ double newton_quotient(double f, double df) {
  const double adf = fabs(df);
  if (!(adf > 1e-30 && adf < 1e30)) return f / df;
  return f * (double)__frcp_rn(__double2float_rn(df));
}

// One real root of q inside the bracket [a, b] (f(a), f(b) of opposite sign, q monotone there):
// Newton's iteration started from the regula-falsi point of the bracket (the ends' values are
// known, and the brackets are narrow: one grid cell or one monotone segment), kept inside the
// shrinking bracket by a bisection step whenever Newton would leave it.  Stops after a step of
// relative size <= 1e-8 (quadratic convergence: the error is then ~1e-16).  The oracle's fast
// formulation runs the same operations.
__device__ __forceinline__ double bracket_root(const double* q, int nq, double a, double b, double fa, double fb) {
  if (fa == 0.0) return a;
  if (fb == 0.0) return b;
  double xl = fa < 0.0 ? a : b, xh = fa < 0.0 ? b : a;  // f(xl) < 0 < f(xh)
  double x = a - fa * newton_quotient(b - a, fb - fa);
  if (!(x > fmin(a, b) && x < fmax(a, b))) x = 0.5 * (a + b);
  for (int it = 0; it < 100; ++it) {
    double f, df;
    horner2(q, nq, x, &f, &df);
    if (f == 0.0) return x;
    if (f < 0.0) xl = x; else xh = x;
    double dx = newton_quotient(f, df);
    double xn = x - dx;
    if (xn == x) return x;  // converged to the last bit (checked before the bracket test: x itself is one end of the bracket)
    if (!(xn >= fmin(xl, xh) && xn <= fmax(xl, xh))) {  // Newton leaves the bracket (or is not finite): bisect
      xn = 0.5 * (xl + xh);
      dx = x - xn;
    }
    if (xn == x) return x;
    x = xn;
    if (fabs(dx) <= 1e-8 * fabs(x)) return x;
  }
  return x;
}

// Roots of q (nq coefficients) in the segments cut out of [lo, hi] by its sorted
// critical points brk[0..nbrk) (nbrk <= 3): q is monotone on each segment, so a
// sign change brackets exactly one root.  One segment per lane; the results are
// gathered in segment order (ascending), dropping repeats.
__device__ __forceinline__ int segment_roots(const double* q, int nq, double b0, double b1, double b2, int nbrk,
                                             double lo, double hi, double* out, int lane) {
  bool has = false;
  double r = 0.0;
  if (lane <= nbrk) {
    const double lefts[4] = {lo, b0, b1, b2};
    const double xa = lane == 0 ? lefts[0] : (lane == 1 ? lefts[1] : (lane == 2 ? lefts[2] : lefts[3]));
    const double inner = lane == 0 ? b0 : (lane == 1 ? b1 : b2);
    const double xb = (lane < nbrk) ? inner : hi;
    double fa, fb, tmp;
    horner2(q, nq, xa, &fa, &tmp);
    horner2(q, nq, xb, &fb, &tmp);
    has = ((fa <= 0.0 && fb >= 0.0) || (fa >= 0.0 && fb <= 0.0)) && !(fa == 0.0 && fb == 0.0);
    if (has) r = bracket_root(q, nq, xa, xb, fa, fb);
  }
  int cnt = 0;
  for (int s = 0; s <= nbrk; ++s) {
    const int hs = __shfl_sync(0xffffffffu, (int)has, s);
    const double rs = __shfl_sync(0xffffffffu, r, s);
    if (hs && (cnt == 0 || rs != out[cnt - 1])) out[cnt++] = rs;
  }
  return cnt;
}

// Real roots inside [lo, hi] of a polynomial of degree <= 3, ascending.
// Degree <= 2: the closed forms of Ceres' polynomial.cc.
__device__ __forceinline__ int roots_upto3(const double* c, int n, double lo, double hi, double* out, int lane) {
  int lead = 0;
  while (lead + 1 < n && c[lead] == 0.0) ++lead;   // RemoveLeadingZeros
  const double* p = c + lead;
  const int degree = n - lead - 1;
  if (degree <= 0) return 0;
  int cnt = 0;
  if (degree == 1) {
    const double r = -p[1] / p[0];
    if (r >= lo && r <= hi) out[cnt++] = r;
    return cnt;
  }
  if (degree == 2) {  // FindQuadraticPolynomialRoots, real case
    const double a = p[0], b = p[1], cc = p[2];
    const double D = b * b - 4 * a * cc;
    if (D < 0) return 0;
    const double sq = sqrt(D);
    double r0, r1;
    if (b >= 0) {
      r0 = (-b - sq) / (2.0 * a);
      r1 = (2.0 * cc) / (-b - sq);
    } else {
      r0 = (2.0 * cc) / (-b + sq);
      r1 = (-b + sq) / (2.0 * a);
    }
    if (r1 < r0) { const double t = r0; r0 = r1; r1 = t; }
    if (r0 >= lo && r0 <= hi) out[cnt++] = r0;
    if (r1 >= lo && r1 <= hi && r1 != r0) out[cnt++] = r1;
    return cnt;
  }
  const double d[3] = {3.0 * p[0], 2.0 * p[1], p[2]};  // critical points of the cubic
  double crit[2] = {0.0, 0.0};
  const int ncrit = roots_upto3(d, 3, lo, hi, crit, lane);
  return segment_roots(p, 4, crit[0], crit[1], 0.0, ncrit, lo, hi, out, lane);
}

// Real roots of c[0..n-1] (highest degree first, degree <= 4) inside [lo, hi], ascending.
__device__ __noinline__ int real_roots_in(const double* c, int n, double lo, double hi, double* out, int lane) {
  int lead = 0;
  while (lead + 1 < n && c[lead] == 0.0) ++lead;
  if (n - lead - 1 <= 3) return roots_upto3(c + lead, n - lead, lo, hi, out, lane);
  const double* p = c + lead;  // quartic
  const double d[4] = {4.0 * p[0], 3.0 * p[1], 2.0 * p[2], p[3]};
  double crit[3] = {0.0, 0.0, 0.0};
  const int ncrit = roots_upto3(d, 4, lo, hi, crit, lane);
  return segment_roots(p, 5, crit[0], crit[1], crit[2], ncrit, lo, hi, out, lane);
}

// ---- fixed-degree variants ----------------------------------------------------
// The same operations in the same order as the generic routines above, with the
// sizes known at compile time so that every coefficient and root stays in a
// register (the generic ones index small arrays dynamically -> local memory on
// the critical path of every Newton step).  Used when no leading coefficient
// vanishes; the generic routines remain the fallback.
template <int N>
__device__ __forceinline__ void horner2_n(const double (&q)[N], double x, double* f, double* df) {
  double v = q[0], d = 0.0;
#pragma unroll
  for (int i = 1; i < N; ++i) {
    d = d * x + v;
    v = v * x + q[i];
  }
  *f = v;
  *df = d;
}

template <int N>
__device__ __forceinline__ double poly_eval_n(const double (&p)[N], double x) {
  double v = 0.0;
#pragma unroll
  for (int i = 0; i < N; ++i) v = v * x + p[i];
  return v;
}

template <int N>
__device__ __forceinline__ double bracket_root_n(const double (&q)[N], double a, double b, double fa, double fb) {
  if (fa == 0.0) return a;
  if (fb == 0.0) return b;
  double xl = fa < 0.0 ? a : b, xh = fa < 0.0 ? b : a;
  double x = a - fa * newton_quotient(b - a, fb - fa);
  if (!(x > fmin(a, b) && x < fmax(a, b))) x = 0.5 * (a + b);
  for (int it = 0; it < 100; ++it) {
    double f, df;
    horner2_n<N>(q, x, &f, &df);
    if (f == 0.0) return x;
    if (f < 0.0) xl = x; else xh = x;
    double dx = newton_quotient(f, df);
    double xn = x - dx;
    if (xn == x) return x;  // converged to the last bit (checked before the bracket test: x itself is one end of the bracket)
    if (!(xn >= fmin(xl, xh) && xn <= fmax(xl, xh))) {
      xn = 0.5 * (xl + xh);
      dx = x - xn;
    }
    if (xn == x) return x;
    x = xn;
    if (fabs(dx) <= 1e-8 * fabs(x)) return x;
  }
  return x;
}

// segment_roots with N coefficients and at most M segments (M = N - 2)
template <int N, int M>
__device__ __forceinline__ int segment_roots_n(const double (&q)[N], double b0, double b1, double b2, int nbrk,
                                               double lo, double hi, double (&out)[M], int lane) {
  bool has = false;
  double r = 0.0;
  if (lane <= nbrk) {
    const double xa = lane == 0 ? lo : (lane == 1 ? b0 : (lane == 2 ? b1 : b2));
    const double inner = lane == 0 ? b0 : (lane == 1 ? b1 : b2);
    const double xb = (lane < nbrk) ? inner : hi;
    double fa, fb, tmp;
    horner2_n<N>(q, xa, &fa, &tmp);
    horner2_n<N>(q, xb, &fb, &tmp);
    has = ((fa <= 0.0 && fb >= 0.0) || (fa >= 0.0 && fb <= 0.0)) && !(fa == 0.0 && fb == 0.0);
    if (has) r = bracket_root_n<N>(q, xa, xb, fa, fb);
  }
  int cnt = 0;
  double last = 0.0;
#pragma unroll
  for (int s = 0; s < M; ++s) {
    const int hs = __shfl_sync(0xffffffffu, (int)has, s);
    const double rs = __shfl_sync(0xffffffffu, r, s);
    if (s <= nbrk && hs && (cnt == 0 || rs != last)) {
#pragma unroll
      for (int k = 0; k < M; ++k)
        if (cnt == k) out[k] = rs;
      last = rs;
      ++cnt;
    }
  }
  return cnt;
}

// FindQuadraticPolynomialRoots, real case, a != 0; roots inside [lo, hi], ascending
__device__ __forceinline__ int quadratic_roots_in(double a, double b, double cc, double lo, double hi, double* o0,
                                                  double* o1) {
  const double D = b * b - 4 * a * cc;
  if (D < 0) return 0;
  const double sq = sqrt(D);
  double r0, r1;
  if (b >= 0) {
    r0 = (-b - sq) / (2.0 * a);
    r1 = (2.0 * cc) / (-b - sq);
  } else {
    r0 = (2.0 * cc) / (-b + sq);
    r1 = (-b + sq) / (2.0 * a);
  }
  if (r1 < r0) { const double t = r0; r0 = r1; r1 = t; }
  int cnt = 0;
  if (r0 >= lo && r0 <= hi) { *o0 = r0; cnt = 1; }
  if (r1 >= lo && r1 <= hi && r1 != r0) {
    if (cnt == 0) *o0 = r1; else *o1 = r1;
    ++cnt;
  }
  return cnt;
}

// Real roots in [lo, hi] of the quartic q (q[0] != 0), ascending
__device__ __forceinline__ int quartic_roots_in(const double (&q)[5], double lo, double hi, double (&out)[4], int lane) {
  const double d3[4] = {4.0 * q[0], 3.0 * q[1], 2.0 * q[2], q[3]};
  double c0 = 0.0, c1 = 0.0;
  const int n2 = quadratic_roots_in(3.0 * d3[0], 2.0 * d3[1], d3[2], lo, hi, &c0, &c1);
  double crit[3] = {0.0, 0.0, 0.0};
  const int n3 = segment_roots_n<4, 3>(d3, c0, c1, 0.0, n2, lo, hi, crit, lane);
  const int n4 = segment_roots_n<5, 4>(q, crit[0], crit[1], crit[2], n3, lo, hi, out, lane);
  return n4;
}

// ---- Budan-Fourier grid isolation of the quartic's roots ----------------------
// The derivative recursion above runs three dependent stages (quadratic, cubic,
// quartic) with a handful of lanes.  Here all 32 lanes work at once: lane L takes
// the grid point t_L = lo + L (hi - lo) / 31 and computes the Taylor coefficients
// of q there (q, q', q"/2, q(3)/6, q(4)/24) by repeated synthetic division.
// With V(t) = number of sign variations of that sequence, Budan-Fourier says the
// number of roots of q in (t_L, t_L+1] is D = V(t_L) - V(t_L+1) minus an even
// number.  So a cell with
//   D = 0                 has no root,
//   D = 1                 has exactly one (q changes sign across it),
//   D = 2, D' = 0         has none   (D' = the same count for q': q is monotone),
//   D = 2, D' = 1         has none or two: q has exactly one extremum e in the
//                         cell (bracketed by the sign change of q'), and the sign
//                         of q(e) decides; the two roots are then bracketed by
//                         [t_L, e] and [e, t_L+1],
//   D = 3, D' = 0         has exactly one (monotone),
// and every other case (two extrema inside one cell, an exact zero on the grid,
// non-finite values) goes to the derivative recursion, which stays the reference.
// Every root is polished by the same safeguarded Newton as before, from a bracket
// 31x tighter, so both routes return the same roots up to the last bits.
__device__ __forceinline__ int quartic_roots_grid(const double (&q)[5], double lo, double hi, double (&out)[4],
                                                  int lane) {
  const double w = (hi - lo) * (1.0 / 31.0);
  const double t = lane == 31 ? hi : fma(w, (double)lane, lo);
  double a1 = q[1], a2 = q[2], a3 = q[3], a4 = q[4];
  const double a0 = q[0];
  a1 = fma(a0, t, a1); a2 = fma(a1, t, a2); a3 = fma(a2, t, a3); a4 = fma(a3, t, a4);  // a4 = q(t)
  a1 = fma(a0, t, a1); a2 = fma(a1, t, a2); a3 = fma(a2, t, a3);                       // a3 = q'(t)
  a1 = fma(a0, t, a1); a2 = fma(a1, t, a2);                                            // a2 = q"(t) / 2
  a1 = fma(a0, t, a1);                                                                 // a1 = q(3)(t) / 6
  const bool bad = !isfinite(a4) || a4 == 0.0 || a3 == 0.0 || a2 == 0.0 || a1 == 0.0;
  const int n4 = a4 < 0.0, n3 = a3 < 0.0, n2 = a2 < 0.0, n1 = a1 < 0.0, n0 = a0 < 0.0;
  const int Vp = (n3 ^ n2) + (n2 ^ n1) + (n1 ^ n0);
  const int V = (n4 ^ n3) + Vp;
  const int Vn = __shfl_down_sync(0xffffffffu, V, 1), Vpn = __shfl_down_sync(0xffffffffu, Vp, 1);
  const double tn = __shfl_down_sync(0xffffffffu, t, 1);
  const double qn = __shfl_down_sync(0xffffffffu, a4, 1), dqn = __shfl_down_sync(0xffffffffu, a3, 1);
  int kind = 0;  // 0 no root, 1 one root in [t, tn], 2 one extremum to examine, 3 undecided
  if (lane < 31) {
    const int D = V - Vn, Dp = Vp - Vpn;
    if (D < 0 || Dp < 0 || D > 3) kind = 3;
    else if (D == 1) kind = 1;
    else if (D == 2) kind = Dp == 0 ? 0 : (Dp == 1 ? 2 : 3);
    else if (D == 3) kind = Dp == 0 ? 1 : 3;
  }
  if (__any_sync(0xffffffffu, bad || kind == 3)) return quartic_roots_in(q, lo, hi, out, lane);
  // cells with one extremum of q: find it, look at the sign of q there
  int nl = kind == 1 ? 1 : 0;
  double xb = tn, fb = qn, e = 0.0, qe = 0.0;
  if (__any_sync(0xffffffffu, kind == 2)) {
    if (kind == 2) {
      const double d3[4] = {4.0 * q[0], 3.0 * q[1], 2.0 * q[2], q[3]};
      e = bracket_root_n<4>(d3, t, tn, a3, dqn);
      qe = poly_eval_n<5>(q, e);
      if (qe != 0.0 && ((qe < 0.0) != (a4 < 0.0))) {  // q crosses zero on both sides of e
        nl = 2;
        xb = e;
        fb = qe;
      }
    }
  }
  double ra = 0.0, rb = 0.0;
  if (nl >= 1) ra = bracket_root_n<5>(q, t, xb, a4, fb);
  if (__any_sync(0xffffffffu, nl == 2)) {
    if (nl == 2) rb = bracket_root_n<5>(q, e, tn, qe, qn);
  }
  // gather in ascending order (cells are ordered, ra < rb inside a cell)
  unsigned m1 = __ballot_sync(0xffffffffu, nl >= 1);
  const unsigned m2 = __ballot_sync(0xffffffffu, nl == 2);
  int cnt = 0;
  double last = 0.0;
  while (m1) {
    const int L = __ffs(m1) - 1;
    m1 &= m1 - 1;
    const double r1 = __shfl_sync(0xffffffffu, ra, L), r2 = __shfl_sync(0xffffffffu, rb, L);
#pragma unroll
    for (int rep = 0; rep < 2; ++rep) {
      const double r = rep == 0 ? r1 : r2;
      if ((rep == 0 || ((m2 >> L) & 1u)) && cnt < 4 && (cnt == 0 || r != last)) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (cnt == k) out[k] = r;
        last = r;
        ++cnt;
      }
    }
  }
  return cnt;
}

// Minimiser over [lo, hi] (in x) of the Hermite interpolant through (0, f0, g0),
// (x1, f1, g1) [and (x2, f2, g2) if three == true].  Warp-uniform.
__device__ __noinline__ double hermite_minimizer(double f0, double g0, double x1, double f1, double g1,
                                                 bool three, double x2, double f2, double g2, double lo,
                                                 double hi, int lane) {
  const double h = three ? fmax(x1, x2) : x1;
  const double ih = 1.0 / h;  // the only division by h: t = x * ih
  const double g0h = g0 * h;
  double c[6];
  int nc;
  if (!three) {
    const double u = f1 - f0 - g0h, v = (g1 - g0) * h;
    c[0] = v - 2.0 * u;
    c[1] = 3.0 * u - v;
    c[2] = g0h;
    c[3] = f0;
    nc = 4;
  } else {
    // p(t) = f0 + g0h t + t^2 s(t): s is the cubic Hermite interpolant of
    // S = (p - f0 - g0h t) / t^2 and its derivative D at ta and tb, in Newton's
    // divided differences, expanded to monomials: three independent reciprocals
    // instead of the four dependent pivots of a 4x4 elimination
    const double ta = x1 * ih, tb = x2 * ih;
    const double ita = 1.0 / ta, itb = 1.0 / tb, iw = 1.0 / (tb - ta);
    const double ita2 = ita * ita, itb2 = itb * itb;
    const double Sa = (f1 - f0 - g0h * ta) * ita2;
    const double Sb = (f2 - f0 - g0h * tb) * itb2;
    const double Da = ((g1 - g0) * h - 2.0 * ta * Sa) * ita2;
    const double Db = ((g2 - g0) * h - 2.0 * tb * Sb) * itb2;
    const double m = (Sb - Sa) * iw;
    const double e2 = (m - Da) * iw;
    const double e3 = ((Db - m) - (m - Da)) * iw * iw;
    c[0] = e3;
    c[1] = e2 - e3 * (2.0 * ta + tb);
    c[2] = Da + ta * (e3 * (ta + 2.0 * tb) - 2.0 * e2);
    c[3] = Sa + ta * (ta * (e2 - e3 * tb) - Da);
    c[4] = g0h;
    c[5] = f0;
    nc = 6;
  }
  const double tlo = lo * ih, thi = hi * ih;
  const double sx[3] = {0.0, x1, x2};
  if (three && c[0] != 0.0) {
    // quintic with a full-degree derivative: everything in registers
    const double c6[6] = {c[0], c[1], c[2], c[3], c[4], c[5]};
    double ox = (lo + hi) / 2.0;
    double ov = poly_eval_n<6>(c6, ox * ih);
    double v = poly_eval_n<6>(c6, tlo);
    if (v < ov) { ov = v; ox = lo; }
    v = poly_eval_n<6>(c6, thi);
    if (v < ov) { ov = v; ox = hi; }
    const double der4[5] = {5.0 * c6[0], 4.0 * c6[1], 3.0 * c6[2], 2.0 * c6[3], c6[4]};
    double roots[4] = {0.0, 0.0, 0.0, 0.0};
    const int nr = quartic_roots_grid(der4, tlo, thi, roots, lane);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i < nr && roots[i] >= tlo && roots[i] <= thi) {
        v = poly_eval_n<6>(c6, roots[i]);
        if (v < ov) { ov = v; ox = roots[i] * h; }
      }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      if (sx[i] >= lo && sx[i] <= hi) {
        v = poly_eval_n<6>(c6, sx[i] * ih);
        if (v < ov) { ov = v; ox = sx[i]; }
      }
    }
    return ox;
  }
  if (!three && c[0] != 0.0) {
    // cubic: the derivative is a quadratic with closed-form roots
    const double c4[4] = {c[0], c[1], c[2], c[3]};
    double ox = (lo + hi) / 2.0;
    double ov = poly_eval_n<4>(c4, ox * ih);
    double v = poly_eval_n<4>(c4, tlo);
    if (v < ov) { ov = v; ox = lo; }
    v = poly_eval_n<4>(c4, thi);
    if (v < ov) { ov = v; ox = hi; }
    double r0 = 0.0, r1 = 0.0;
    const int nr = quadratic_roots_in(3.0 * c4[0], 2.0 * c4[1], c4[2], tlo, thi, &r0, &r1);
    if (nr > 0) {
      v = poly_eval_n<4>(c4, r0);
      if (v < ov) { ov = v; ox = r0 * h; }
    }
    if (nr > 1) {
      v = poly_eval_n<4>(c4, r1);
      if (v < ov) { ov = v; ox = r1 * h; }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      if (sx[i] >= lo && sx[i] <= hi) {
        v = poly_eval_n<4>(c4, sx[i] * ih);
        if (v < ov) { ov = v; ox = sx[i]; }
      }
    }
    return ox;
  }
  // MinimizePolynomial: middle, ends, real parts of the roots of p'
  double ox = (lo + hi) / 2.0;
  double ov = poly_eval(c, nc, ox * ih);
  double v = poly_eval(c, nc, tlo);
  if (v < ov) { ov = v; ox = lo; }
  v = poly_eval(c, nc, thi);
  if (v < ov) { ov = v; ox = hi; }
  double der[5], roots[4];
  const int degree = nc - 1;
  for (int i = 0; i < degree; ++i) der[i] = (degree - i) * c[i];
  const int nr = real_roots_in(der, degree, tlo, thi, roots, lane);
  for (int i = 0; i < nr; ++i) {
    if (roots[i] < tlo || roots[i] > thi) continue;
    v = poly_eval(c, nc, roots[i]);
    if (v < ov) { ov = v; ox = roots[i] * h; }
  }
  // MinimizeInterpolatingPolynomial: the samples themselves, in order
  for (int i = 0; i < (three ? 3 : 2); ++i) {
    if (sx[i] < lo || sx[i] > hi) continue;
    v = poly_eval(c, nc, sx[i] * ih);
    if (v < ov) { ov = v; ox = sx[i]; }
  }
  return ox;
}

// One contraction of ArmijoLineSearch::DoSearch: new trial step from
// {initial, current [, previous]}.
__device__ __forceinline__ double ls_next_step(const LsSample& initial, const LsSample& previous,
                                               const LsSample& current, const DevConsts& K, int lane) {
  const double min_step = K.ls_max_contraction * current.x;
  const double max_step = K.ls_min_contraction * current.x;
  // invalid value (or a non-finite gradient, which only overflow can produce):
  // Ceres' bisection rule
  if (!current.value_valid || !current.gradient_valid ||
      (previous.value_valid && !previous.gradient_valid))
    return fmin(fmax(current.x * 0.5, min_step), max_step);
  return hermite_minimizer(initial.value, initial.gradient, current.x, current.value, current.gradient,
                           previous.value_valid, previous.x, previous.value, previous.gradient, min_step,
                           max_step, lane);
}

// warp-wide helpers --------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}

}  // namespace lfr
