/* ekf_device.cuh -- device-side arithmetic shared by ekf_kernels.cu and ekf_batch.cu.
 *
 * Every function restates, operation for operation, the scalar expansion of the GSL reference-BLAS loop
 * that slam_ros/Robot.cpp calls at the cited line (SURVEY.md appendix A).  The explicit round-to-nearest
 * intrinsics are never contracted into FMAs.
 */
#ifndef EKF_DEVICE_CUH
#define EKF_DEVICE_CUH
#include <math.h>

#define EKF_PI 3.14159265358979323846

__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
/* acc += t*b as the reference-BLAS NN/TN loops do it.  Those loops skip a term whose multiplier t is exactly zero; for
 * finite b the skipped update acc + 0*b leaves acc bit for bit unchanged (only a zero acc can change sign), so the
 * test-and-select is not issued: on B200 a DSETP + select in a dependent chain costs 18 cycles against 8 for the plain
 * DMUL / DADD (profiles/r2_fp64_latency.log), and these chains ARE the per-line latency.  -DEKF_ZERO_SKIP restores the
 * literal skip (it only differs when the covariance already holds Inf / NaN). */
#ifdef EKF_ZERO_SKIP
#define EKF_NZ(t) ((t) != 0.0)
#else
#define EKF_NZ(t) true
#endif
__device__ __forceinline__ void axpy_skip(double& acc, double t, double b) {
  if (EKF_NZ(t)) acc = add_rn(acc, mul_rn(t, b));
}
/* cos and sin of one angle.  sincos() shares the argument reduction between the two and returns the SAME bits as cos() and
 * sin() called separately (checked on the device: 200 scans at 1k landmarks, state and covariance bit-equal); on the gate's
 * dependent chain that is ~1.5 % of a step at 1k landmarks and of a Monte-Carlo batch step.  -DEKF_SEPARATE_SINCOS restores
 * the two calls. */
__device__ __forceinline__ void cos_sin(double x, double& c, double& s) {
#ifdef EKF_SEPARATE_SINCOS
  c = cos(x); s = sin(x);
#else
  sincos(x, &s, &c);
#endif
}
/* one rank-2 term of Robot.cpp:564:  (0 + ks.x*k.x) + ks.y*k.y  */
__device__ __forceinline__ double rank2(double2 ks, double2 k) {
  return add_rn(mul_rn(ks.x, k.x), mul_rn(ks.y, k.y));
}

/* p - (ks.x*k.x + ks.y*k.y): the per-element update of Robot.cpp:564-568.
 * Default: two fused multiply-adds, p <- fma(-ks.y, k.y, fma(-ks.x, k.x, p)).  The reference (x86-64 GSL, no
 * FMA) rounds ks.x*k.x, ks.y*k.y, their sum and the difference separately; the fused form differs from that by
 * at most a few ulp of the products (orders of magnitude inside the 1e-9 bar) and halves the fp64 issue
 * slots, which is what keeps the rank-2m sweep HBM-bound at m = 8.  Every kernel uses this one function, so
 * all launch strategies stay bit-identical to each other.  -DEKF_EXACT_RANK2 restores the reference order. */
__device__ __forceinline__ double sub_rank2(double p, double2 ks, double2 k) {
#ifdef EKF_EXACT_RANK2
  return sub_rn(p, rank2(ks, k));
#else
  return __fma_rn(-ks.y, k.y, __fma_rn(-ks.x, k.x, p));
#endif
}

/* Robot.cpp:62-71 verbatim (C++ parses floor(..)*2.0*M_PI as (floor(..)*2.0)*M_PI) */
__device__ __forceinline__ void normalize_radian(double& rad) {
  const double two_pi = 2.0 * EKF_PI;
  if (rad > EKF_PI) {
    const double f = floor(__ddiv_rn(rad, two_pi));
    rad = sub_rn(rad, add_rn(two_pi, mul_rn(mul_rn(f, 2.0), EKF_PI)));
  } else if (rad < -EKF_PI) {
    const double f = floor(__ddiv_rn(fabs(rad), two_pi));
    rad = add_rn(rad, add_rn(two_pi, mul_rn(mul_rn(f, 2.0), EKF_PI)));
  }
}

struct Gate {
  double c, s, g;
  double S[4], Si[4];
  double v[2];
  double d2;
  int singular;
};

/* gsl_linalg_LU_decomp + LU_invert on a 2x2 (Robot.cpp:431-457); GSL <= 2.5 unblocked order */
__device__ __forceinline__ int inv2x2_lu(const double S[4], double Si[4]) {
  double a0 = S[0], a1 = S[1], a2 = S[2], a3 = S[3];
  int p0 = 0, p1 = 1;
  if (fabs(a2) > fabs(a0)) { double t = a0; a0 = a2; a2 = t; t = a1; a1 = a3; a3 = t; p0 = 1; p1 = 0; }
  if (a0 != 0.0) {
    const double l = __ddiv_rn(a2, a0);
    a2 = l;
    a3 = sub_rn(a3, mul_rn(l, a1));
  }
  if (a0 == 0.0 || a3 == 0.0) { Si[0] = Si[1] = Si[2] = Si[3] = 0.0; return 1; }
  for (int col = 0; col < 2; ++col) {
    double x0 = (p0 == col) ? 1.0 : 0.0;
    double x1 = (p1 == col) ? 1.0 : 0.0;
    x1 = sub_rn(x1, mul_rn(a2, x0));
    x1 = __ddiv_rn(x1, a3);
    x0 = __ddiv_rn(sub_rn(x0, mul_rn(a1, x1)), a0);
    Si[col] = x0; Si[2 + col] = x1;
  }
  return 0;
}

/* The D x D generalisation of inv2x2_lu (D <= 3, row stride 3): gsl_linalg_LU_decomp (first-largest partial pivot,
 * elimination skipped on a zero pivot) then gsl_linalg_LU_invert, one column of the identity at a time: permute, unit
 * lower forward substitution, upper back substitution, in the reference-BLAS dtrsv order.  Returns 1 (Si = 0) when a
 * diagonal entry of U is zero, as LU_invert's singularity test does. */
template <int D>
__device__ __forceinline__ int invDxD_lu(const double S[9], double Si[9]) {
  double a[D][D];
  int p[D];
#pragma unroll
  for (int i = 0; i < D; ++i) {
    p[i] = i;
#pragma unroll
    for (int k = 0; k < D; ++k) a[i][k] = S[3 * i + k];
  }
#pragma unroll
  for (int j = 0; j < D - 1; ++j) {
    double mx = fabs(a[j][j]);
    int piv = j;
#pragma unroll
    for (int i = j + 1; i < D; ++i) if (fabs(a[i][j]) > mx) { mx = fabs(a[i][j]); piv = i; }
#pragma unroll
    for (int i = j + 1; i < D; ++i)             /* swap rows j and piv (register arrays: select, no dynamic index) */
      if (piv == i) {
#pragma unroll
        for (int k = 0; k < D; ++k) { const double t = a[j][k]; a[j][k] = a[i][k]; a[i][k] = t; }
        const int t = p[j]; p[j] = p[i]; p[i] = t;
      }
    const double ajj = a[j][j];
    if (ajj != 0.0) {
#pragma unroll
      for (int i = j + 1; i < D; ++i) {
        const double l = __ddiv_rn(a[i][j], ajj);
        a[i][j] = l;
#pragma unroll
        for (int k = j + 1; k < D; ++k) a[i][k] = sub_rn(a[i][k], mul_rn(l, a[j][k]));
      }
    }
  }
  bool sing = false;
#pragma unroll
  for (int i = 0; i < D; ++i) sing = sing || a[i][i] == 0.0;
  if (sing) {
#pragma unroll
    for (int t = 0; t < 9; ++t) Si[t] = 0.0;
    return 1;
  }
#pragma unroll
  for (int col = 0; col < D; ++col) {
    double x[D];
#pragma unroll
    for (int i = 0; i < D; ++i) x[i] = (p[i] == col) ? 1.0 : 0.0;
#pragma unroll
    for (int i = 1; i < D; ++i)                                        /* L x = P e (unit diagonal) */
#pragma unroll
      for (int k = 0; k < i; ++k) x[i] = sub_rn(x[i], mul_rn(a[i][k], x[k]));
    x[D - 1] = __ddiv_rn(x[D - 1], a[D - 1][D - 1]);                   /* U x = . */
#pragma unroll
    for (int i = D - 2; i >= 0; --i) {
      double t = x[i];
#pragma unroll
      for (int k = i + 1; k < D; ++k) t = sub_rn(t, mul_rn(a[i][k], x[k]));
      x[i] = __ddiv_rn(t, a[i][i]);
    }
#pragma unroll
    for (int i = 0; i < D; ++i) Si[3 * i + col] = x[i];
  }
  return 0;
}

/* Robot.cpp:367-489 for one (line, landmark) pair, given P gathered at rows/cols {0,1,2,a,b} (Cm), the
 * landmark (m0, m1) = (y[a], y[b]), the predicted pose, the observed line z and its covariance R.
 *
 * The reference-BLAS loops the reference calls multiply by the structural +-1 entries of H and start every sum from
 * 0.0; those operations are exact (x*1 = x, x*(-1) = -x, 0 + x = x) and are not issued here: every value is bit for bit
 * what the literal sequence produces, except that a zero result may carry the other sign (0.0 + (-0.0) = +0.0), which no
 * comparison, product or sum downstream can tell apart.  What is kept is every operation that rounds, in the
 * reference's order (the zero skips of the NN / TN loops: see axpy_skip). */
__device__ __forceinline__ void gate_from_block(const double Cm[5][5], double m0, double m1, const double x_pre[3],
                                                double z0, double z1, const double R[4], Gate& G) {
  double c, s;
  cos_sin(m0, c, s);
  const double H10 = -c, H11 = -s;
  const double gg = sub_rn(mul_rn(x_pre[0], s), mul_rn(x_pre[1], c));     /* Robot.cpp:379 */
  G.c = c; G.s = s; G.g = gg;
  double HP0[5], HP1[5];
#pragma unroll
  for (int t = 0; t < 5; ++t) {                                       /* :397  H * P  (NN, k = 0,1,2,a,b) */
    double h1 = EKF_NZ(H10) ? mul_rn(H10, Cm[0][t]) : 0.0;
    axpy_skip(h1, H11, Cm[1][t]);
    axpy_skip(h1, gg, Cm[3][t]);
    h1 = add_rn(h1, Cm[4][t]);
    HP0[t] = sub_rn(Cm[3][t], Cm[2][t]);                              /* (0 + -P[2,t]) + P[a,t] */
    HP1[t] = h1;
  }
#pragma unroll
  for (int p = 0; p < 2; ++p) {                                       /* :401  HP * H'  (NT) */
    const double* HP = p ? HP1 : HP0;
    double t1 = mul_rn(HP[0], H10);
    t1 = add_rn(t1, mul_rn(HP[1], H11));
    t1 = add_rn(t1, mul_rn(HP[3], gg));
    t1 = add_rn(t1, HP[4]);
    G.S[p * 2 + 0] = sub_rn(HP[3], HP[2]);
    G.S[p * 2 + 1] = t1;
  }
#pragma unroll
  for (int t = 0; t < 4; ++t) G.S[t] = add_rn(G.S[t], R[t]);            /* :405 */
  double h0 = sub_rn(m0, x_pre[2]);                                     /* :423-426 */
  const double h1 = sub_rn(m1, add_rn(mul_rn(x_pre[0], c), mul_rn(x_pre[1], s)));
  normalize_radian(h0);
  G.singular = inv2x2_lu(G.S, G.Si);
  double v0 = sub_rn(z0, h0);                                           /* :465 */
  const double v1 = sub_rn(z1, h1);
  const double two_pi = 2.0 * EKF_PI;                                 /* :471-475 */
  if (fabs(sub_rn(v0, two_pi)) < fabs(v0)) v0 = sub_rn(v0, two_pi);
  else if (fabs(add_rn(v0, two_pi)) < fabs(v0)) v0 = add_rn(v0, two_pi);
  G.v[0] = v0; G.v[1] = v1;
  double w0 = 0.0, w1 = 0.0;                                          /* :479  v' * Sinv  (TN) */
  if (EKF_NZ(v0)) { w0 = mul_rn(v0, G.Si[0]); w1 = mul_rn(v0, G.Si[1]); }
  axpy_skip(w0, v1, G.Si[2]); axpy_skip(w1, v1, G.Si[3]);
  double d2 = EKF_NZ(w0) ? mul_rn(w0, v0) : 0.0;                      /* :483 */
  axpy_skip(d2, w1, v1);
  G.d2 = d2;
}

/* gain row r of Robot.cpp:522-560 from the five entries P[r,{0,1,2,a,b}] (exact operations elided as above) */
__device__ __forceinline__ void gain_row(const Gate& G, double p0, double p1, double p2, double pa, double pb,
                                         double2& K, double2& KS) {
  const double H10 = -G.c, H11 = -G.s, gg = G.g;
  const double ph0 = sub_rn(pa, p2);                                  /* :522  P * H'  (NT) */
  double ph1 = mul_rn(p0, H10);
  ph1 = add_rn(ph1, mul_rn(p1, H11));
  ph1 = add_rn(ph1, mul_rn(pa, gg));
  ph1 = add_rn(ph1, pb);
  double k0 = 0.0, k1 = 0.0;                                          /* :526  PHt * Sinv  (NN) */
  if (EKF_NZ(ph0)) { k0 = mul_rn(ph0, G.Si[0]); k1 = mul_rn(ph0, G.Si[1]); }
  axpy_skip(k0, ph1, G.Si[2]); axpy_skip(k1, ph1, G.Si[3]);
  double s0 = 0.0, s1 = 0.0;                                          /* :560  K * S  (NN) */
  if (EKF_NZ(k0)) { s0 = mul_rn(k0, G.S[0]); s1 = mul_rn(k0, G.S[1]); }
  axpy_skip(s0, k1, G.S[2]); axpy_skip(s1, k1, G.S[3]);
  K = make_double2(k0, k1); KS = make_double2(s0, s1);
}

/* Robot.cpp:489 rejects when sqrt(|d2|) > gate.  sqrt is correctly rounded and monotone, so the test is the same as
 * |d2| > T with T the largest double whose square root does not exceed the gate: one comparison instead of the
 * square root's dependent chain.  (NaN: both forms compare false -- the pair passes, as in the reference.) */
__host__ __device__ inline bool gate_rejects_d2(double d2, double d2max) { return fabs(d2) > d2max; }
#endif
